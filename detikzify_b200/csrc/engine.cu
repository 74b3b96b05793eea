// C-ABI implementation (see include/detikzify_b200.h). Host-side orchestration only: weight-arena
// layout, KV sequence slots, workspaces, CUDA-graph capture of the decode+sample step and the launch
// sequences for ViT encode / projector / prefill / decode. All arithmetic is in the .cu kernels.
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "../../include/detikzify_b200.h"
#include "launch.h"

using namespace dtk;

namespace {

struct WEntry {
  std::string name;
  int rows, cols;
  uint64_t offset, nbytes;
};

inline uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }
inline int patch_k_padded(const dtk_config& c) { return (int)align_up((uint64_t)3 * c.v_patch * c.v_patch, 64); }
inline int v_tokens(const dtk_config& c) { int g = c.v_image / c.v_patch; return g * g; }
inline int img_tokens(const dtk_config& c) { return v_tokens(c) / c.concat; }

std::vector<WEntry> build_table(const dtk_config& c) {
  std::vector<WEntry> t;
  uint64_t off = 0;
  auto add = [&](const std::string& n, int rows, int cols) {
    WEntry e{n, rows, cols, off, (uint64_t)rows * cols * 2};
    off = align_up(off + e.nbytes, 256);
    t.push_back(e);
  };
  const int H = c.hidden, I = c.inter, V = c.vocab, qd = c.heads * c.head_dim, kd = c.kv_heads * c.head_dim;
  add("dec.embed", V, H);
  for (int l = 0; l < c.layers; ++l) {
    std::string p = "dec.L" + std::to_string(l) + ".";
    add(p + "norm1", 1, H);
    add(p + "wqkv", qd + 2 * kd, H);
    add(p + "wo", H, qd);
    add(p + "norm2", 1, H);
    add(p + "wgu", 2 * I, H);  // interleaved rows: 2i = gate_i, 2i+1 = up_i
    add(p + "wd", H, I);
  }
  add("dec.norm", 1, H);
  add("dec.lm_head", V, H);
  const int D = c.v_hidden, VI = c.v_inter, N = v_tokens(c);
  add("proj.w", H, D * c.concat);
  add("proj.b", 1, H);
  add("vit.patch_w", D, patch_k_padded(c));
  add("vit.patch_b", 1, D);
  add("vit.pos", N, D);
  for (int l = 0; l < c.v_layers; ++l) {
    std::string p = "vit.L" + std::to_string(l) + ".";
    add(p + "ln1_w", 1, D); add(p + "ln1_b", 1, D);
    add(p + "wqkv", 3 * D, D); add(p + "bqkv", 1, 3 * D);
    add(p + "wo", D, D); add(p + "bo", 1, D);
    add(p + "ln2_w", 1, D); add(p + "ln2_b", 1, D);
    add(p + "w1", VI, D); add(p + "b1", 1, VI);
    add(p + "w2", D, VI); add(p + "b2", 1, D);
  }
  add("vit.post_w", 1, D); add("vit.post_b", 1, D);
  add("vit.head.probe", 1, D);
  add("vit.head.wq", D, D); add("vit.head.bq", 1, D);
  add("vit.head.wkv", 2 * D, D); add("vit.head.bkv", 1, 2 * D);
  add("vit.head.wo", D, D); add("vit.head.bo", 1, D);
  add("vit.head.ln_w", 1, D); add("vit.head.ln_b", 1, D);
  add("vit.head.w1", VI, D); add("vit.head.b1", 1, VI);
  add("vit.head.w2", D, VI); add("vit.head.b2", 1, D);
  return t;
}

bool config_ok(const dtk_config& c, std::string& why) {
  auto bad = [&](const char* m) { why = m; return false; };
  if (c.hidden <= 0 || c.inter <= 0 || c.layers <= 0 || c.heads <= 0 || c.kv_heads <= 0 || c.vocab <= 0) return bad("non-positive decoder dims");
  if (c.head_dim != 128) return bad("decoder head_dim must be 128");
  if (c.heads % c.kv_heads) return bad("heads % kv_heads != 0");
  if ((c.hidden & 7) || (c.inter & 7)) return bad("hidden/inter must be multiples of 8");
  if (c.rope_type != 0 && c.rope_type != 1) return bad("rope_type must be 0 (linear) or 1 (llama3)");
  if (c.rope_type == 1 && (c.rope_low_freq <= 0.f || c.rope_high_freq <= c.rope_low_freq || c.rope_orig_max_pos <= 0)) return bad("bad llama3 rope parameters");
  if (c.max_len <= 0 || c.max_seqs <= 0 || c.max_batch <= 0 || c.max_batch > 64) return bad("bad max_len/max_seqs/max_batch (max_batch <= 64)");
  if (c.v_hidden <= 0 || c.v_heads <= 0 || c.v_hidden % c.v_heads) return bad("bad vision dims");
  if (c.v_hidden / c.v_heads != 72) return bad("vision head_dim must be 72 (SigLIP so400m)");
  if ((c.v_hidden & 7) || (c.v_inter & 7)) return bad("vision dims must be multiples of 8");
  if (c.v_patch <= 0 || c.v_image < c.v_patch) return bad("bad image/patch size");  // conv stride P, no padding: floor(S/P) patches
  if (c.concat <= 0 || img_tokens(c) <= 0) return bad("bad concat");
  return true;
}

}  // namespace

struct dtk_engine {
  dtk_config cfg;
  int device = 0;
  std::string err;
  uint64_t launches = 0;
  const uint8_t* arena = nullptr;
  std::map<std::string, const bf16*> w;

  // KV slots: [slot][layer][2][kv_head][max_len][128] bf16
  bf16* kv = nullptr;
  int64_t kv_layer_stride = 0, kv_v_offset = 0, kv_slot_stride = 0;
  std::vector<char> slot_used;
  // one-level shared KV prefix: positions [0, share_len[s]) of slot s are read from slot share_base[s] (a multiple of 16
  // positions, never written through s); refcnt[b] = sequences borrowing from b, shared_upto[b] = longest prefix lent out
  std::vector<int> share_base, share_len, refcnt, shared_upto;
  float* rope_cs = nullptr;  // [max_len, 64, 2]

  // prefill workspace (max_len rows)
  float *p_x = nullptr, *p_qkv = nullptr;
  bf16 *p_xn = nullptr, *p_q = nullptr, *p_att = nullptr, *p_h = nullptr;
  // decode workspace (max_batch rows)
  float *d_x = nullptr, *d_q = nullptr, *d_att = nullptr, *d_h = nullptr, *d_logits = nullptr, *d_scratch = nullptr;
  float *d_part_o = nullptr, *d_part_ml = nullptr;
  unsigned int* d_counters = nullptr;  // [max_batch*heads] + 1 (sampler done counter)
  int *d_slots = nullptr, *d_pos = nullptr, *d_tok = nullptr, *d_share_slot = nullptr, *d_share_len = nullptr;
  unsigned long long* d_gen = nullptr;  // [0] = step counter
  // ViT workspace (grows with batch)
  int vit_cap = 0;
  float *v_x = nullptr, *v_small_f = nullptr, *v_pq = nullptr;
  bf16 *v_xn = nullptr, *v_qkv = nullptr, *v_att = nullptr, *v_h = nullptr, *v_small_b = nullptr;
  bool pq_ready = false;
  // the ViT forward of a chunk of nb images is captured once per (nb, outputs) into a CUDA graph over engine-owned
  // staging buffers (~250 launches per chunk, each encoding two tensor maps on the host, become one graph launch)
  struct VitGraph { cudaGraphExec_t exec; uint64_t launches; };
  std::map<int, VitGraph> vit_graphs;
  float *v_pix_in = nullptr, *v_tok_out = nullptr, *v_pool_out = nullptr;
  bf16* v_vt = nullptr;      // per-layer V^T copy for the tcgen05 attention
  int vit_graph = 1;
  int attn_impl = 1;         // ViT attention: 1 = tcgen05 (attn_tc.cu), 0 = mma.sync flash attention (attn_mma.cu)

  // generation loop
  int gen_B = 0;
  dtk_sampling gen_params{};
  unsigned long long* host_ring = nullptr;   // pinned, mapped: [ring][64] entries ((step + 1) << 32) | token
  unsigned long long* dev_ring = nullptr;
  int ring = 256;
  std::map<std::string, cudaGraphExec_t> graphs;
  cudaGraphExec_t gen_graph = nullptr;
  cudaStream_t gen_stream = nullptr;
  cudaStream_t cap_stream = nullptr;  // engine-owned: graph capture never touches the caller's stream
  // persistent decode kernel (B = 1)
  MegaArgs mega{};
  int mega_grid = 0;
  bool mega_ok = false;
  int decode_impl = 1;       // 1 = persistent weight-streaming kernel (default), 0 = per-op kernels / CUDA graph
  int decode_gemm_min_batch = 4;  // B >= this: batched decode runs the dense matrices as tensor-core GEMMs (weights once per step)
  bool gen_mega = false;
  bool gen_fused = false;    // greedy generation on the persistent kernel: argmax + token publication in the kernel tail
  unsigned long long* d_amax = nullptr;
  SampleArgs gen_sample{};
  unsigned long long* d_bar = nullptr;  // [0] counter, [1] epoch base
  unsigned int* d_head_cnt = nullptr;
  bf16* d_tiled = nullptr;             // decode-side re-tiled copy of the decoder matrices
  unsigned long long* d_tagged = nullptr;  // {fp32 value, phase tag} cross-CTA activation words of the persistent kernel
  long long* d_dbg = nullptr;           // phase timestamps of the persistent kernel (option mega_debug)
  long long* d_dbg2 = nullptr;          // per-tile clock trace of one layer (option mega_trace_layer)
  int mega_trace_layer = -1;
  int mega_debug = 0;
  int mega_flags = 0;
  int mega_variant = 0;
  int mega_nslots = 0;       // dev option "mega_nslots": cap on the ring depth of the persistent kernel (0 = as configured)
  int fuse_greedy = 1;
  int cascade_attn = 1;      // batched decode: rows that share one prefix reduce it with ONE tensor-core pass (option "cascade_attn")
  int cas_slot = -1, cas_len = 0;   // set per step by dtk_decode / dtk_gen_begin: uniform shared prefix of the current batch
};

namespace {

#define DTK_CK(expr)                                                                          \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      eng->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                          \
      return DTK_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define DTK_REQUIRE(cond, msg)                                                                \
  do {                                                                                        \
    if (!(cond)) {                                                                            \
      eng->err = std::string("invalid argument: ") + msg;                                     \
      return DTK_ERR_INVALID;                                                                 \
    }                                                                                         \
  } while (0)

template <typename T>
int dev_alloc(dtk_engine* eng, T** p, uint64_t count) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T));
  if (e != cudaSuccess) {
    eng->err = std::string("cudaMalloc failed: ") + cudaGetErrorString(e);
    cudaGetLastError();
    return DTK_ERR_OOM;
  }
  *p = (T*)q;
  return DTK_OK;
}
#define DTK_ALLOC(ptr, count)                         \
  do {                                                \
    int _r = dev_alloc(eng, &(ptr), (uint64_t)(count)); \
    if (_r != DTK_OK) return _r;                      \
  } while (0)

const bf16* W(dtk_engine* eng, const std::string& n) { return eng->w.at(n); }
std::string LN(const char* prefix, int l, const char* s) { return std::string(prefix) + std::to_string(l) + "." + s; }

struct StateArgs {
  int n;
  int slots[64], pos[64], share_slot[64], share_len[64];
  long long tok[64];
  int have_tok;
};
__global__ void set_state_kernel(StateArgs a, int* slots, int* pos, int* tok, int* share_slot, int* share_len) {
  int i = threadIdx.x;
  if (i < a.n) {
    slots[i] = a.slots[i];
    pos[i] = a.pos[i];
    share_slot[i] = a.share_slot[i];
    share_len[i] = a.share_len[i];
    if (a.have_tok) tok[i] = (int)a.tok[i];
  }
}
// rows of a batched step that all borrow the same prefix [0, len) from the same slot (the rollouts of one figure)
void set_cascade(dtk_engine* eng, const StateArgs& st) {
  eng->cas_slot = -1; eng->cas_len = 0;
  if (!eng->cascade_attn || st.n < 4 || st.n > 64) return;
  const int len = st.share_len[0], base = st.share_slot[0];
  if (len < 64 || base == st.slots[0]) return;
  for (int i = 1; i < st.n; ++i)
    if (st.share_len[i] != len || st.share_slot[i] != base) return;
  eng->cas_slot = base; eng->cas_len = len;
}
__global__ void tok64_to_32_kernel(const int64_t* in, int* out, int n) {
  if ((int)threadIdx.x < n) out[threadIdx.x] = (int)in[threadIdx.x];
}
__global__ void reset_gen_kernel(unsigned long long* gen, unsigned int* done, unsigned long long seed) {
  gen[0] = 0ull;
  gen[1] = seed;   // read by the sampler of the generation loop (not baked into the captured graph)
  *done = 0u;
}

constexpr int VIT_CHUNK = 64;   // images per ViT pass (larger batches are processed in chunks)

// ViT workspace: allocated ONCE, for a full chunk, at the first vision call (no regrowth: a cudaFree inside a stream-ordered
// call would synchronise the device, and captured graphs keep pointing at these buffers)
int ensure_vit_ws(dtk_engine* eng, int /*B*/) {
  if (eng->vit_cap > 0) return DTK_OK;
  const dtk_config& c = eng->cfg;
  const int B = VIT_CHUNK;
  const int64_t rows = (int64_t)B * v_tokens(c);
  DTK_ALLOC(eng->v_x, rows * c.v_hidden);
  DTK_ALLOC(eng->v_xn, rows * c.v_hidden);
  DTK_ALLOC(eng->v_qkv, rows * 3 * c.v_hidden);
  DTK_ALLOC(eng->v_att, rows * c.v_hidden);
  int64_t hcols = c.v_inter > patch_k_padded(c) ? c.v_inter : patch_k_padded(c);
  DTK_ALLOC(eng->v_h, rows * hcols);
  DTK_ALLOC(eng->v_small_f, (int64_t)B * c.v_hidden * 2);
  DTK_ALLOC(eng->v_small_b, (int64_t)B * (c.v_hidden * 2 + c.v_inter));
  DTK_ALLOC(eng->v_pix_in, (int64_t)B * 3 * c.v_image * c.v_image);
  DTK_ALLOC(eng->v_tok_out, rows * c.v_hidden);
  DTK_ALLOC(eng->v_pool_out, (int64_t)B * c.v_hidden);
  DTK_ALLOC(eng->v_vt, (int64_t)B * c.v_heads * 80 * attn_tc_vt_cols(v_tokens(c)));
  eng->vit_cap = B;
  return DTK_OK;
}

// probe query of the attention-pool head: input independent (q = probe Wq^T + bq), computed once per engine
int ensure_probe_query(dtk_engine* eng, cudaStream_t s) {
  if (eng->pq_ready) return DTK_OK;
  const int D = eng->cfg.v_hidden;
  GemmArgs g{};
  g.A = W(eng, "vit.head.probe"); g.lda = D; g.W = W(eng, "vit.head.wq"); g.ldw = D; g.M = 1; g.N = D; g.K = D;
  g.bias = W(eng, "vit.head.bq"); g.out_f32 = eng->v_pq; g.ldo = D;
  DTK_CK(launch_gemm(g, s, &eng->launches));
  eng->pq_ready = true;
  return DTK_OK;
}

// ViT blocks for B images already resident as fp32 pixels; leaves post-LN tokens (bf16) in v_xn.
int vit_forward(dtk_engine* eng, const float* pixels, int B, float* tokens_out, float* pooled_out, cudaStream_t s) {
  const dtk_config& c = eng->cfg;
  const int D = c.v_hidden, VI = c.v_inter, N = v_tokens(c), KP = patch_k_padded(c);
  const int M = B * N;
  const int act = c.v_act == 1 ? ACT_GELU_ERF : ACT_GELU_TANH;
  uint64_t* lc = &eng->launches;
  bf16* col = eng->v_h;  // alias: v_h is free until the first MLP
  DTK_CK(launch_im2col(pixels, B, c.v_image, c.v_patch, KP, col, s, lc));
  {
    GemmArgs g{};
    g.A = col; g.lda = KP; g.W = W(eng, "vit.patch_w"); g.ldw = KP; g.M = M; g.N = D; g.K = KP;
    g.bias = W(eng, "vit.patch_b"); g.rowbias = W(eng, "vit.pos"); g.rowbias_mod = N;
    g.out_f32 = eng->v_x; g.ldo = D;
    DTK_CK(launch_gemm(g, s, lc));
  }
  for (int l = 0; l < c.v_layers; ++l) {
    DTK_CK(launch_layernorm(eng->v_x, W(eng, LN("vit.L", l, "ln1_w")), W(eng, LN("vit.L", l, "ln1_b")), c.v_eps, M, D, eng->v_xn, nullptr, s, lc));
    {
      GemmArgs g{};
      g.A = eng->v_xn; g.lda = D; g.W = W(eng, LN("vit.L", l, "wqkv")); g.ldw = D; g.M = M; g.N = 3 * D; g.K = D;
      g.bias = W(eng, LN("vit.L", l, "bqkv")); g.out_bf16 = eng->v_qkv; g.ldo = 3 * D;
      DTK_CK(launch_gemm(g, s, lc));
    }
    if (eng->attn_impl == 1 && attn_tc_supported()) {
      DTK_CK(launch_attn_tc(eng->v_qkv, eng->v_vt, eng->v_att, B, c.v_heads, N, 1.0f / sqrtf(72.f), s, lc));
    } else {
      AttnArgs a{};
      a.q = eng->v_qkv; a.k = eng->v_qkv + D; a.v = eng->v_qkv + 2 * D; a.o = eng->v_att;
      a.q_bs = a.k_bs = a.v_bs = (int64_t)N * 3 * D; a.q_hs = a.k_hs = a.v_hs = 72; a.q_rs = a.k_rs = a.v_rs = 3 * D;
      a.o_bs = (int64_t)N * D; a.o_hs = 72; a.o_rs = D;
      a.B = B; a.heads = c.v_heads; a.kv_group = 1; a.Tq = N; a.Tk = N; a.q_pos0 = 0; a.causal = 0; a.head_dim = 72;
      a.scale = 1.0f / sqrtf(72.f);
      DTK_CK(launch_flash_attn(a, s, lc));
    }
    {
      GemmArgs g{};
      g.A = eng->v_att; g.lda = D; g.W = W(eng, LN("vit.L", l, "wo")); g.ldw = D; g.M = M; g.N = D; g.K = D;
      g.bias = W(eng, LN("vit.L", l, "bo")); g.resid = eng->v_x; g.ldr = D; g.out_f32 = eng->v_x; g.ldo = D;
      DTK_CK(launch_gemm(g, s, lc));
    }
    DTK_CK(launch_layernorm(eng->v_x, W(eng, LN("vit.L", l, "ln2_w")), W(eng, LN("vit.L", l, "ln2_b")), c.v_eps, M, D, eng->v_xn, nullptr, s, lc));
    {
      GemmArgs g{};
      g.A = eng->v_xn; g.lda = D; g.W = W(eng, LN("vit.L", l, "w1")); g.ldw = D; g.M = M; g.N = VI; g.K = D;
      g.bias = W(eng, LN("vit.L", l, "b1")); g.act = act; g.out_bf16 = eng->v_h; g.ldo = VI;
      DTK_CK(launch_gemm(g, s, lc));
    }
    {
      GemmArgs g{};
      g.A = eng->v_h; g.lda = VI; g.W = W(eng, LN("vit.L", l, "w2")); g.ldw = VI; g.M = M; g.N = D; g.K = VI;
      g.bias = W(eng, LN("vit.L", l, "b2")); g.resid = eng->v_x; g.ldr = D; g.out_f32 = eng->v_x; g.ldo = D;
      DTK_CK(launch_gemm(g, s, lc));
    }
  }
  DTK_CK(launch_layernorm(eng->v_x, W(eng, "vit.post_w"), W(eng, "vit.post_b"), c.v_eps, M, D, eng->v_xn, tokens_out, s, lc));

  if (pooled_out) {
    bf16* kvb = eng->v_qkv;  // [M, 2D]
    {
      GemmArgs g{};
      g.A = eng->v_xn; g.lda = D; g.W = W(eng, "vit.head.wkv"); g.ldw = D; g.M = M; g.N = 2 * D; g.K = D;
      g.bias = W(eng, "vit.head.bkv"); g.out_bf16 = kvb; g.ldo = 2 * D;
      DTK_CK(launch_gemm(g, s, lc));
    }
    bf16* pa = eng->v_small_b;               // [B, D] attention output
    bf16* pn = eng->v_small_b + (int64_t)B * D;      // [B, D] LN output
    bf16* ph = eng->v_small_b + (int64_t)B * 2 * D;  // [B, VI]
    float* pr = eng->v_small_f;              // [B, D] residual
    DTK_CK(launch_pool_attn(eng->v_pq, kvb, B, N, D, c.v_heads, 1.0f / sqrtf(72.f), pa, s, lc));
    {
      GemmArgs g{};
      g.A = pa; g.lda = D; g.W = W(eng, "vit.head.wo"); g.ldw = D; g.M = B; g.N = D; g.K = D;
      g.bias = W(eng, "vit.head.bo"); g.out_f32 = pr; g.ldo = D;
      DTK_CK(launch_gemm(g, s, lc));
    }
    DTK_CK(launch_layernorm(pr, W(eng, "vit.head.ln_w"), W(eng, "vit.head.ln_b"), c.v_eps, B, D, pn, nullptr, s, lc));
    {
      GemmArgs g{};
      g.A = pn; g.lda = D; g.W = W(eng, "vit.head.w1"); g.ldw = D; g.M = B; g.N = VI; g.K = D;
      g.bias = W(eng, "vit.head.b1"); g.act = act; g.out_bf16 = ph; g.ldo = VI;
      DTK_CK(launch_gemm(g, s, lc));
    }
    {
      GemmArgs g{};
      g.A = ph; g.lda = VI; g.W = W(eng, "vit.head.w2"); g.ldw = VI; g.M = B; g.N = D; g.K = VI;
      g.bias = W(eng, "vit.head.b2"); g.resid = pr; g.ldr = D; g.out_f32 = pooled_out; g.ldo = D;
      DTK_CK(launch_gemm(g, s, lc));
    }
  }
  return DTK_OK;
}

// concat-3 projector on bf16 tokens [B, N, D] -> fp32 [B, P, H]
int project_bf16(dtk_engine* eng, const bf16* tokens, int B, float* out, cudaStream_t s) {
  const dtk_config& c = eng->cfg;
  const int D = c.v_hidden, N = v_tokens(c), P = img_tokens(c), K = D * c.concat;
  GemmArgs g{};
  g.A = tokens + (int64_t)(N - P * c.concat) * D;  // drop the first patches when N % concat != 0
  g.lda = K; g.a_rows_per_batch = P; g.a_batch_stride = (int64_t)N * D;
  g.W = W(eng, "proj.w"); g.ldw = K; g.M = B * P; g.N = c.hidden; g.K = K;
  g.bias = W(eng, "proj.b"); g.out_f32 = out; g.ldo = c.hidden;
  DTK_CK(launch_gemm(g, s, &eng->launches));
  return DTK_OK;
}

bf16* kv_layer(dtk_engine* eng, int slot, int layer) {
  return eng->kv + (int64_t)slot * eng->kv_slot_stride + (int64_t)layer * eng->kv_layer_stride;
}

int nsplit_for(const dtk_config& c, int B) {
  int n = (2 * 148 + c.heads * B - 1) / (c.heads * B);
  if (n < 1) n = 1;
  if (n > 16) n = 16;
  return n;
}

// one decode step for the B sequences whose (slot, pos, tok) live in d_slots / d_pos / d_tok (or tok64)
int decode_launches(dtk_engine* eng, int B, const int64_t* tok64, float* logits, cudaStream_t s) {
  const dtk_config& c = eng->cfg;
  const int H = c.hidden, I = c.inter, qd = c.heads * 128, kd = c.kv_heads * 128;
  uint64_t* lc = &eng->launches;
  if (B == 1 && eng->decode_impl == 1 && eng->mega_ok) {
    if (tok64) {
      tok64_to_32_kernel<<<1, 32, 0, s>>>(tok64, eng->d_tok, 1);
      ++*lc;
      DTK_CK(cudaGetLastError());
    }
    MegaArgs m = eng->mega;
    m.logits = logits;
    m.dbg = eng->mega_debug ? eng->d_dbg : nullptr;
    m.dbg_flags = eng->mega_flags;
    m.variant = eng->mega_variant;
    if (eng->mega_nslots >= 8 && eng->mega_nslots < m.nslots) m.nslots = eng->mega_nslots & ~7;
    m.fuse_greedy = 0;
    if (eng->gen_fused && logits == eng->d_logits) {   // inside the greedy generation loop
      m.fuse_greedy = 1; m.bad_token = eng->gen_sample.bad_token; m.ring = eng->ring; m.max_pos = eng->cfg.max_len - 1;
      m.amax = eng->d_amax; m.gen_tok = eng->d_tok; m.gen_pos = eng->d_pos; m.gen_step = eng->d_gen; m.host_ring = eng->dev_ring;
    }
    m.dbg2 = (eng->mega_debug && eng->mega_trace_layer >= 0) ? eng->d_dbg2 : nullptr;
    m.dbg_layer = eng->mega_trace_layer;
    DTK_CK(launch_decode_mega(m, eng->mega_grid, s, lc));
    return DTK_OK;
  }
  DTK_CK(launch_embed_tokens(tok64 ? nullptr : eng->d_tok, tok64, B, W(eng, "dec.embed"), H, c.vocab, eng->d_x, s, lc));
  int nsplit = nsplit_for(c, B);
  if (eng->decode_gemm_min_batch > 0 && B >= eng->decode_gemm_min_batch && B <= c.max_len) {
    if (eng->cas_len > 0 && eng->cas_slot >= 0 && nsplit > 4) nsplit = 4;   // cascade: the per-row kernel covers the (short) private suffix only; 12+ partial slots stay for the prefix   // (B rows fit the prefill buffers)
    // ---- batched decode (MCTS rollouts / several figures): the B rows go through the dense matrices as ONE GEMM each, so
    // the weights are streamed once per step instead of once per sequence (the GEMV kernels below re-read them B times:
    // measured 59 ms/step for 32 ds-7b rollouts). Activations are rounded to bf16 GEMM operands exactly as in prefill
    // (fp32 residual stream, fp32 accumulation); RoPE / KV append / attention are per row (slot, position).
    const int qkvd = qd + 2 * kd;
    auto gemm = [&](const bf16* A, int K, const bf16* Wm, int N, const float* resid, int glu, float* o32, bf16* o16, int ldo) {
      GemmArgs g{};
      g.A = A; g.lda = K; g.W = Wm; g.ldw = K; g.M = B; g.N = N; g.K = K;
      g.resid = resid; g.ldr = ldo; g.glu = glu; g.out_f32 = o32; g.out_bf16 = o16; g.ldo = ldo;
      return launch_gemm(g, s, lc);
    };
    // Shared-prefix ("cascade") attention: when every row borrows the same prefix from one slot (MCTS rollouts of a figure),
    // the prefix keys are reduced ONCE per head by the tensor-core flash kernel with the B query rows as its M dimension
    // (K/V tiles read once instead of B times: 60 -> ~10 us per ds-7b layer at 32 rollouts x 500 shared positions); the
    // per-row kernel covers the private suffix only and merges both partial sets.
    const bool cas = eng->cas_len > 0 && eng->cas_slot >= 0;
    const int ctiles_all = cas ? (eng->cas_len + 63) / 64 : 0;
    const int cslots = 16 - nsplit;   // partial slots per (row, head) left for the prefix (buffers hold 16)
    const int ctile = cas ? std::max(2, (ctiles_all + cslots - 1) / cslots) : 0;   // 64-key tiles per prefix CTA
    const int csplit = cas ? (ctiles_all + ctile - 1) / ctile : 0;
    for (int l = 0; l < c.layers; ++l) {
      DTK_CK(launch_rmsnorm(eng->d_x, H, W(eng, LN("dec.L", l, "norm1")), c.rms_eps, B, H, eng->p_xn, s, lc));
      DTK_CK(gemm(eng->p_xn, H, W(eng, LN("dec.L", l, "wqkv")), qkvd, nullptr, 0, eng->p_qkv, nullptr, qkvd));
      DTK_CK(launch_rope_kv_decode(eng->p_qkv, B, eng->d_slots, eng->d_pos, c.heads, c.kv_heads, eng->rope_cs, eng->d_q,
                                   kv_layer(eng, 0, l), eng->kv_slot_stride, eng->kv_v_offset, c.max_len, s, lc, cas ? eng->p_q : nullptr));
      if (cas) {
        AttnArgs f{};
        f.q = eng->p_q; f.k = kv_layer(eng, eng->cas_slot, l); f.v = f.k + eng->kv_v_offset;
        f.q_bs = 0; f.q_hs = 128; f.q_rs = qd;
        f.k_bs = 0; f.k_hs = (int64_t)c.max_len * 128; f.k_rs = 128;
        f.v_bs = 0; f.v_hs = (int64_t)c.max_len * 128; f.v_rs = 128;
        f.B = 1; f.heads = c.heads; f.kv_group = c.heads / c.kv_heads; f.Tq = B; f.Tk = eng->cas_len; f.q_pos0 = 0;
        f.causal = 0; f.head_dim = 128; f.scale = 1.0f / sqrtf(128.f);
        f.part_o = eng->d_part_o; f.part_ml = eng->d_part_ml; f.part_np = nsplit + csplit; f.part_idx0 = nsplit; f.part_tiles = ctile;
        DTK_CK(launch_flash_attn(f, s, lc));
      }
      {
        DecodeAttnArgs a{};
        a.q = eng->d_q; a.q_stride = qd; a.kv_base = kv_layer(eng, 0, l); a.kv_slot_stride = eng->kv_slot_stride;
        a.kv_v_offset = eng->kv_v_offset; a.slots = eng->d_slots; a.pos = eng->d_pos; a.share_slot = eng->d_share_slot; a.share_len = eng->d_share_len;
        a.B = B; a.heads = c.heads; a.kv_group = c.heads / c.kv_heads; a.max_len = c.max_len; a.nsplit = nsplit;
        a.scale = 1.0f / sqrtf(128.f);
        a.part_o = eng->d_part_o; a.part_ml = eng->d_part_ml; a.counters = eng->d_counters;
        a.out = eng->d_att; a.out_stride = qd; a.out_bf16 = eng->p_att;   // bf16 copy = the o-proj operand (no cast launch)
        if (cas) { a.key_begin = eng->cas_len; a.np = nsplit + csplit; }
        DTK_CK(launch_decode_attn(a, s, lc));
      }
      DTK_CK(gemm(eng->p_att, qd, W(eng, LN("dec.L", l, "wo")), H, eng->d_x, 0, eng->d_x, nullptr, H));
      DTK_CK(launch_rmsnorm(eng->d_x, H, W(eng, LN("dec.L", l, "norm2")), c.rms_eps, B, H, eng->p_xn, s, lc));
      DTK_CK(gemm(eng->p_xn, H, W(eng, LN("dec.L", l, "wgu")), 2 * I, nullptr, 1, nullptr, eng->p_h, I));
      DTK_CK(gemm(eng->p_h, I, W(eng, LN("dec.L", l, "wd")), H, eng->d_x, 0, eng->d_x, nullptr, H));
    }
    DTK_CK(launch_rmsnorm(eng->d_x, H, W(eng, "dec.norm"), c.rms_eps, B, H, eng->p_xn, s, lc));
    DTK_CK(gemm(eng->p_xn, H, W(eng, "dec.lm_head"), c.vocab, nullptr, 0, logits, nullptr, c.vocab));
    return DTK_OK;
  }
  for (int l = 0; l < c.layers; ++l) {
    {
      GemvArgs g{};
      g.mode = GEMV_QKV; g.W = W(eng, LN("dec.L", l, "wqkv")); g.N = qd + 2 * kd; g.K = H;
      g.x = eng->d_x; g.x_stride = H; g.norm_w = W(eng, LN("dec.L", l, "norm1")); g.eps = c.rms_eps;
      g.out = eng->d_q; g.out_stride = qd; g.B = B;
      g.slots = eng->d_slots; g.pos = eng->d_pos; g.rope_cs = eng->rope_cs;
      g.kv_base = kv_layer(eng, 0, l); g.kv_slot_stride = eng->kv_slot_stride; g.kv_v_offset = eng->kv_v_offset;
      g.q_dim = qd; g.kv_dim = kd; g.max_len = c.max_len;
      DTK_CK(launch_gemv(g, s, lc));
    }
    {
      DecodeAttnArgs a{};
      a.q = eng->d_q; a.q_stride = qd; a.kv_base = kv_layer(eng, 0, l); a.kv_slot_stride = eng->kv_slot_stride;
      a.kv_v_offset = eng->kv_v_offset; a.slots = eng->d_slots; a.pos = eng->d_pos; a.share_slot = eng->d_share_slot; a.share_len = eng->d_share_len;
      a.B = B; a.heads = c.heads; a.kv_group = c.heads / c.kv_heads; a.max_len = c.max_len; a.nsplit = nsplit;
      a.scale = 1.0f / sqrtf(128.f);
      a.part_o = eng->d_part_o; a.part_ml = eng->d_part_ml; a.counters = eng->d_counters;
      a.out = eng->d_att; a.out_stride = qd;
      DTK_CK(launch_decode_attn(a, s, lc));
    }
    {
      GemvArgs g{};
      g.mode = GEMV_ADD; g.W = W(eng, LN("dec.L", l, "wo")); g.N = H; g.K = qd;
      g.x = eng->d_att; g.x_stride = qd; g.out = eng->d_x; g.out_stride = H; g.B = B;
      DTK_CK(launch_gemv(g, s, lc));
    }
    {
      GemvArgs g{};
      g.mode = GEMV_GLU; g.W = W(eng, LN("dec.L", l, "wgu")); g.N = 2 * I; g.K = H;
      g.x = eng->d_x; g.x_stride = H; g.norm_w = W(eng, LN("dec.L", l, "norm2")); g.eps = c.rms_eps;
      g.out = eng->d_h; g.out_stride = I; g.B = B;
      DTK_CK(launch_gemv(g, s, lc));
    }
    {
      GemvArgs g{};
      g.mode = GEMV_ADD; g.W = W(eng, LN("dec.L", l, "wd")); g.N = H; g.K = I;
      g.x = eng->d_h; g.x_stride = I; g.out = eng->d_x; g.out_stride = H; g.B = B;
      DTK_CK(launch_gemv(g, s, lc));
    }
  }
  {
    GemvArgs g{};
    g.mode = GEMV_STORE; g.W = W(eng, "dec.lm_head"); g.N = c.vocab; g.K = H;
    g.x = eng->d_x; g.x_stride = H; g.norm_w = W(eng, "dec.norm"); g.eps = c.rms_eps;
    g.out = logits; g.out_stride = c.vocab; g.B = B;
    DTK_CK(launch_gemv(g, s, lc));
  }
  return DTK_OK;
}

void fill_sample_args(dtk_engine* eng, SampleArgs& a, const float* logits, int B, const dtk_sampling& p) {
  std::memset(&a, 0, sizeof(a));
  a.logits = logits; a.B = B; a.V = eng->cfg.vocab;
  a.temperature = (float)p.temperature; a.top_p = (float)p.top_p; a.top_p_limit = (float)(1.0 - p.top_p); a.top_k = p.top_k;
  a.max_pos = eng->cfg.max_len - 1;
  a.do_sample = (p.do_sample && p.temperature >= 1e-5) ? 1 : 0;
  a.bad_token = p.bad_token; a.bs_token = p.begin_suppress_token; a.seed = p.seed;
  a.scratch = eng->d_scratch;
}

}  // namespace

// ================================================================== C ABI
extern "C" {

int dtk_abi_version(void) { return DTK_ABI_VERSION; }

int dtk_weight_count(const dtk_config* cfg) {
  if (!cfg) return DTK_ERR_INVALID;
  std::string why;
  if (!config_ok(*cfg, why)) return DTK_ERR_INVALID;
  return (int)build_table(*cfg).size();
}

int dtk_weight_get(const dtk_config* cfg, int index, dtk_weight_info* out) {
  if (!cfg || !out) return DTK_ERR_INVALID;
  std::string why;
  if (!config_ok(*cfg, why)) return DTK_ERR_INVALID;
  auto t = build_table(*cfg);
  if (index < 0 || index >= (int)t.size()) return DTK_ERR_INVALID;
  std::memset(out, 0, sizeof(*out));
  std::snprintf(out->name, sizeof(out->name), "%s", t[index].name.c_str());
  out->offset = t[index].offset; out->nbytes = t[index].nbytes; out->rows = t[index].rows; out->cols = t[index].cols;
  return DTK_OK;
}

uint64_t dtk_arena_bytes(const dtk_config* cfg) {
  if (!cfg) return 0;
  std::string why;
  if (!config_ok(*cfg, why)) return 0;
  auto t = build_table(*cfg);
  return align_up(t.back().offset + t.back().nbytes, 256);
}

uint64_t dtk_decode_bytes(const dtk_config* c, int T) {
  if (!c) return 0;
  const uint64_t H = c->hidden, I = c->inter, V = c->vocab, qd = (uint64_t)c->heads * c->head_dim, kd = (uint64_t)c->kv_heads * c->head_dim;
  uint64_t wbytes = 2 * ((uint64_t)c->layers * ((qd + 2 * kd) * H + H * qd + 3 * H * I) + V * H);
  uint64_t kv = 2 * (uint64_t)c->layers * 2 * kd;  // bytes per cached position (K and V, bf16)
  return wbytes + (uint64_t)T * kv;
}

int dtk_create(const dtk_config* cfg, const void* weight_arena, uint64_t arena_bytes, int device, dtk_engine** out) {
  if (!cfg || !weight_arena || !out) return DTK_ERR_INVALID;
  std::string why;
  if (!config_ok(*cfg, why)) return DTK_ERR_INVALID;
  if (arena_bytes < dtk_arena_bytes(cfg)) return DTK_ERR_INVALID;
  dtk_engine* eng = new (std::nothrow) dtk_engine();
  if (!eng) return DTK_ERR_OOM;
  eng->cfg = *cfg;
  eng->device = device;
  *out = eng;  // returned even on failure so the caller can read dtk_last_error, then dtk_destroy
  DTK_CK(cudaSetDevice(device));
  eng->arena = (const uint8_t*)weight_arena;
  for (auto& e : build_table(*cfg)) eng->w[e.name] = (const bf16*)(eng->arena + e.offset);

  const dtk_config& c = eng->cfg;
  const int64_t H = c.hidden, I = c.inter, V = c.vocab, qd = c.heads * 128, kd = c.kv_heads * 128, T = c.max_len, MB = c.max_batch;
  eng->kv_v_offset = (int64_t)c.kv_heads * c.max_len * 128;
  eng->kv_layer_stride = 2 * eng->kv_v_offset;
  eng->kv_slot_stride = eng->kv_layer_stride * c.layers;
  DTK_ALLOC(eng->kv, eng->kv_slot_stride * c.max_seqs);
  eng->slot_used.assign(c.max_seqs, 0);
  eng->share_base.assign(c.max_seqs, -1);
  eng->share_len.assign(c.max_seqs, 0);
  eng->refcnt.assign(c.max_seqs, 0);
  eng->shared_upto.assign(c.max_seqs, 0);

  // RoPE table (HF modeling_llama.py:83-121: inv_freq = theta^(-2i/d) / factor, fp32; angle = pos * inv_freq)
  {
    std::vector<float> tab((size_t)T * 64 * 2);
    for (int i = 0; i < 64; ++i) {
      float inv = 1.0f / powf(c.rope_theta, (float)(2 * i) / 128.0f);
      if (c.rope_type == 1) {   // llama3 (HF modeling_rope_utils.py _compute_llama3_parameters), fp32 like HF
        const float old_len = (float)c.rope_orig_max_pos;
        const float low_wl = old_len / c.rope_low_freq, high_wl = old_len / c.rope_high_freq;
        const float wl = 2.0f * 3.14159265358979323846f / inv;
        if (wl > low_wl) inv = inv / c.rope_factor;
        else if (!(wl < high_wl)) {
          const float smooth = (old_len / wl - c.rope_low_freq) / (c.rope_high_freq - c.rope_low_freq);
          inv = (1.0f - smooth) * inv / c.rope_factor + smooth * inv;
        }
      } else {
        inv = inv / c.rope_factor;
      }
      for (int64_t p = 0; p < T; ++p) {
        float ang = (float)p * inv;
        tab[((size_t)p * 64 + i) * 2] = (float)cos((double)ang);
        tab[((size_t)p * 64 + i) * 2 + 1] = (float)sin((double)ang);
      }
    }
    DTK_ALLOC(eng->rope_cs, tab.size());
    DTK_CK(cudaMemcpy(eng->rope_cs, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  DTK_ALLOC(eng->p_x, T * H);
  DTK_ALLOC(eng->p_qkv, T * (qd + 2 * kd));
  DTK_ALLOC(eng->p_xn, T * H);
  DTK_ALLOC(eng->p_q, T * qd);
  DTK_ALLOC(eng->p_att, T * qd);
  DTK_ALLOC(eng->p_h, T * I);
  DTK_ALLOC(eng->d_x, MB * H);
  DTK_ALLOC(eng->d_q, MB * qd);
  DTK_ALLOC(eng->d_att, MB * qd);
  DTK_ALLOC(eng->d_h, MB * I);
  DTK_ALLOC(eng->d_logits, MB * V);
  DTK_ALLOC(eng->d_scratch, MB * V);
  DTK_ALLOC(eng->d_part_o, MB * c.heads * 16 * 128);
  DTK_ALLOC(eng->d_part_ml, MB * c.heads * 16 * 2);
  DTK_ALLOC(eng->d_counters, MB * c.heads + 1);
  DTK_CK(cudaMemset(eng->d_counters, 0, (MB * c.heads + 1) * sizeof(unsigned int)));
  DTK_ALLOC(eng->d_slots, MB);
  DTK_ALLOC(eng->d_pos, MB);
  DTK_ALLOC(eng->d_tok, MB);
  DTK_ALLOC(eng->d_share_slot, MB);
  DTK_ALLOC(eng->d_share_len, MB);
  DTK_CK(cudaMemset(eng->d_share_slot, 0, MB * sizeof(int)));
  DTK_CK(cudaMemset(eng->d_share_len, 0, MB * sizeof(int)));
  DTK_ALLOC(eng->d_gen, 2);
  DTK_CK(cudaMemset(eng->d_gen, 0, 2 * sizeof(unsigned long long)));
  DTK_ALLOC(eng->v_pq, c.v_hidden);
  {
    int smem_optin = 0, sms = 0, coop = 0;
    DTK_CK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    DTK_CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    DTK_CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
    MegaArgs& m = eng->mega;
    int grid = 0;
    if (coop && mega_configure(m, c.hidden, c.inter, c.heads, smem_optin, sms, &grid) == cudaSuccess) {
      m.H = c.hidden; m.I = c.inter; m.L = c.layers; m.heads = c.heads; m.kv_heads = c.kv_heads; m.V = c.vocab;
      m.max_len = c.max_len; m.eps = c.rms_eps;
      m.embed = W(eng, "dec.embed"); m.final_norm = W(eng, "dec.norm");
      m.norm1_0 = W(eng, "dec.L0.norm1"); m.norm2_0 = W(eng, "dec.L0.norm2");
      m.norm_stride = c.layers > 1 ? (int64_t)(W(eng, "dec.L1.norm1") - W(eng, "dec.L0.norm1")) : 0;
      // decode-side tiled weight copy (one-time, on device): [layer][qkv | o | gu | down] ... [lm_head]
      const int qkvN = (c.heads + 2 * c.kv_heads) * 128, qd = c.heads * 128;
      struct Spec { MegaMat* mm; const char* name; int N, K, mode; } specs[4] = {
          {&m.mat[0], "wqkv", qkvN, c.hidden, TILE_ROPE}, {&m.mat[1], "wo", c.hidden, qd, TILE_SEQ},
          {&m.mat[2], "wgu", 2 * c.inter, c.hidden, TILE_GLU}, {&m.mat[3], "wd", c.hidden, c.inter, TILE_SEQ}};
      int64_t per_layer = 0, off[4];
      for (int i = 0; i < 4; ++i) {
        off[i] = per_layer;
        per_layer += mega_tiled_elems(specs[i].N, specs[i].K, specs[i].mode, &specs[i].mm->groups, &specs[i].mm->tpg);
      }
      const int64_t lm_elems = mega_tiled_elems(c.vocab, c.hidden, TILE_SEQ, &m.mat[4].groups, &m.mat[4].tpg);
      DTK_ALLOC(eng->d_tiled, per_layer * c.layers + lm_elems);
      for (int i = 0; i < 4; ++i) {
        MegaMat& mm = *specs[i].mm;
        mm.base = eng->d_tiled + off[i]; mm.layer_stride = per_layer; mm.N = specs[i].N; mm.K = specs[i].K; mm.mode = specs[i].mode;
        for (int l = 0; l < c.layers; ++l)
          DTK_CK(launch_retile(W(eng, LN("dec.L", l, specs[i].name)), specs[i].N, specs[i].K, specs[i].mode,
                               eng->d_tiled + (int64_t)l * per_layer + off[i], 0));
      }
      for (int i = 0; i < 5; ++i) {
        m.mat[i].per = (m.mat[i].groups + grid - 1) / grid;
        m.mat[i].nact = (m.mat[i].groups + m.mat[i].per - 1) / m.mat[i].per;
      }
      m.mat[4].base = eng->d_tiled + per_layer * c.layers; m.mat[4].layer_stride = 0; m.mat[4].N = c.vocab; m.mat[4].K = c.hidden; m.mat[4].mode = TILE_SEQ;
      DTK_CK(launch_retile(W(eng, "dec.lm_head"), c.vocab, c.hidden, TILE_SEQ, eng->d_tiled + per_layer * c.layers, 0));
      m.tok = eng->d_tok; m.pos = eng->d_pos; m.slots = eng->d_slots; m.share_slot = eng->d_share_slot; m.share_len = eng->d_share_len;
      m.kv = eng->kv; m.kv_slot_stride = eng->kv_slot_stride; m.kv_layer_stride = eng->kv_layer_stride;
      m.kv_v_offset = eng->kv_v_offset; m.rope_cs = eng->rope_cs;
      m.logits = eng->d_logits;
      {
        const int64_t words = 2 * (int64_t)m.tg_H + 2 * (int64_t)qd + 2 * (int64_t)c.kv_heads * 128 + m.tg_I + (int64_t)grid * 132;
        DTK_ALLOC(eng->d_tagged, words);
        DTK_CK(cudaMemset(eng->d_tagged, 0, (size_t)words * sizeof(unsigned long long)));
        m.tg = eng->d_tagged;
      }
      DTK_ALLOC(eng->d_amax, 2);
      DTK_CK(cudaMemset(eng->d_amax, 0, 2 * sizeof(unsigned long long)));
      DTK_ALLOC(eng->d_bar, 4);
      DTK_CK(cudaMemset(eng->d_bar, 0, 4 * sizeof(unsigned long long)));
      m.bar_count = eng->d_bar; m.bar_base = eng->d_bar + 1;
      DTK_ALLOC(eng->d_head_cnt, c.heads);
      DTK_CK(cudaMemset(eng->d_head_cnt, 0, c.heads * sizeof(unsigned int)));
      m.head_cnt = eng->d_head_cnt;
      DTK_ALLOC(eng->d_dbg, (int64_t)grid * (c.layers * 5 + 1) * 4);
      DTK_CK(cudaMemset(eng->d_dbg, 0, (size_t)grid * (c.layers * 5 + 1) * 4 * sizeof(long long)));
      DTK_ALLOC(eng->d_dbg2, (int64_t)grid * MEGA_DBG2_ROWS * 4);
      DTK_CK(cudaMemset(eng->d_dbg2, 0, (size_t)grid * MEGA_DBG2_ROWS * 4 * sizeof(long long)));
      m.dbg = nullptr; m.dbg2 = nullptr; m.dbg_layer = -1;
      eng->mega_grid = grid;
      eng->mega_ok = true;
    }
  }
  DTK_CK(cudaHostAlloc((void**)&eng->host_ring, (size_t)eng->ring * 64 * sizeof(unsigned long long), cudaHostAllocMapped));
  std::memset(eng->host_ring, 0, (size_t)eng->ring * 64 * sizeof(unsigned long long));
  DTK_CK(cudaHostGetDevicePointer((void**)&eng->dev_ring, eng->host_ring, 0));
  DTK_CK(cudaDeviceSynchronize());
  return DTK_OK;
}

int dtk_destroy(dtk_engine* eng) {
  if (!eng) return DTK_ERR_INVALID;
  cudaSetDevice(eng->device);
  cudaDeviceSynchronize();
  for (auto& g : eng->graphs) cudaGraphExecDestroy(g.second);
  for (auto& g : eng->vit_graphs) cudaGraphExecDestroy(g.second.exec);
  void* ptrs[] = {eng->v_pix_in, eng->v_tok_out, eng->v_pool_out, eng->v_vt, eng->kv, eng->rope_cs, eng->p_x, eng->p_qkv, eng->p_xn, eng->p_q, eng->p_att, eng->p_h, eng->d_x, eng->d_q,
                  eng->d_att, eng->d_h, eng->d_logits, eng->d_scratch, eng->d_part_o, eng->d_part_ml, eng->d_counters,
                  eng->d_slots, eng->d_pos, eng->d_tok, eng->d_share_slot, eng->d_share_len, eng->d_gen, eng->d_amax, eng->d_bar, eng->d_dbg, eng->d_dbg2, eng->d_head_cnt, eng->d_tiled, eng->d_tagged, eng->v_x, eng->v_small_f, eng->v_pq, eng->v_xn,
                  eng->v_qkv, eng->v_att, eng->v_h, eng->v_small_b};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (eng->cap_stream) cudaStreamDestroy(eng->cap_stream);
  if (eng->host_ring) cudaFreeHost(eng->host_ring);
  cudaGetLastError();
  delete eng;
  return DTK_OK;
}

const char* dtk_last_error(const dtk_engine* eng) { return eng ? eng->err.c_str() : "null engine"; }
uint64_t dtk_launch_count(const dtk_engine* eng) { return eng ? eng->launches : 0; }

int dtk_vit_encode(dtk_engine* eng, const float* pixels, int B, float* tokens_out, float* pooled_out, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(pixels && B > 0, "pixels/B");
  DTK_CK(cudaSetDevice(eng->device));
  const dtk_config& c = eng->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  int r = ensure_vit_ws(eng, B);
  if (r != DTK_OK) return r;
  if (pooled_out && (r = ensure_probe_query(eng, s)) != DTK_OK) return r;
  const int64_t pix_per = (int64_t)3 * c.v_image * c.v_image, N = v_tokens(c), D = c.v_hidden;
  for (int b0 = 0; b0 < B; b0 += VIT_CHUNK) {
    const int nb = B - b0 < VIT_CHUNK ? B - b0 : VIT_CHUNK;
    float* tok = tokens_out ? tokens_out + b0 * N * D : nullptr;
    float* pool = pooled_out ? pooled_out + (int64_t)b0 * D : nullptr;
    if (!eng->vit_graph) {
      r = vit_forward(eng, pixels + b0 * pix_per, nb, tok, pool, s);
      if (r != DTK_OK) return r;
      continue;
    }
    const int key = nb | (tok ? 1 << 8 : 0) | (pool ? 1 << 9 : 0) | (get_gemm_impl() << 10) | (eng->attn_impl << 12);
    auto it = eng->vit_graphs.find(key);
    if (it == eng->vit_graphs.end()) {
      if (!eng->cap_stream) DTK_CK(cudaStreamCreateWithFlags(&eng->cap_stream, cudaStreamNonBlocking));
      cudaStream_t cs = eng->cap_stream;
      const uint64_t before = eng->launches;
      cudaGraph_t graph = nullptr;
      DTK_CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
      r = vit_forward(eng, eng->v_pix_in, nb, tok ? eng->v_tok_out : nullptr, pool ? eng->v_pool_out : nullptr, cs);
      cudaError_t ce = cudaStreamEndCapture(cs, &graph);
      const uint64_t n = eng->launches - before;
      eng->launches = before;             // captured launches are counted per replay
      if (r != DTK_OK) { if (graph) cudaGraphDestroy(graph); return r; }
      if (ce != cudaSuccess) { eng->err = std::string("cudaStreamEndCapture (ViT): ") + cudaGetErrorString(ce); return DTK_ERR_CUDA; }
      cudaGraphExec_t exec = nullptr;
      DTK_CK(cudaGraphInstantiate(&exec, graph, 0));
      cudaGraphDestroy(graph);
      it = eng->vit_graphs.emplace(key, dtk_engine::VitGraph{exec, n}).first;
    }
    DTK_CK(cudaMemcpyAsync(eng->v_pix_in, pixels + b0 * pix_per, (size_t)nb * pix_per * sizeof(float), cudaMemcpyDeviceToDevice, s));
    DTK_CK(cudaGraphLaunch(it->second.exec, s));
    eng->launches += it->second.launches;
    if (tok) DTK_CK(cudaMemcpyAsync(tok, eng->v_tok_out, (size_t)nb * N * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (pool) DTK_CK(cudaMemcpyAsync(pool, eng->v_pool_out, (size_t)nb * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  return DTK_OK;
}

int dtk_image_preprocess(dtk_engine* eng, const uint8_t* rgb, int h, int w, int S, const int32_t* bounds_h, const int32_t* coef_h,
                         int ksize_h, const int32_t* bounds_v, const int32_t* coef_v, int ksize_v, float rescale,
                         const float* mean3_host, const float* std3_host, uint8_t* tmp, float* out, uint8_t* out_u8, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(rgb && bounds_h && coef_h && bounds_v && coef_v && mean3_host && std3_host && tmp && out, "null pointer");
  DTK_REQUIRE(h > 0 && w > 0 && S > 0 && ksize_h > 0 && ksize_v > 0, "sizes");
  DTK_CK(cudaSetDevice(eng->device));
  DTK_CK(launch_image_preprocess(rgb, h, w, S, bounds_h, coef_h, ksize_h, bounds_v, coef_v, ksize_v, rescale, mean3_host, std3_host,
                                 tmp, out, out_u8, (cudaStream_t)stream, &eng->launches));
  return DTK_OK;
}

int dtk_project(dtk_engine* eng, const float* tokens, int B, float* out, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(tokens && out && B > 0, "tokens/out/B");
  DTK_CK(cudaSetDevice(eng->device));
  const dtk_config& c = eng->cfg;
  const int CH = VIT_CHUNK;
  int r = ensure_vit_ws(eng, B < CH ? B : CH);
  if (r != DTK_OK) return r;
  const int64_t per = (int64_t)v_tokens(c) * c.v_hidden;
  for (int b0 = 0; b0 < B; b0 += CH) {
    int nb = B - b0 < CH ? B - b0 : CH;
    DTK_CK(launch_cast_f32_bf16(tokens + b0 * per, eng->v_xn, nb * per, (cudaStream_t)stream, &eng->launches));
    r = project_bf16(eng, eng->v_xn, nb, out + (int64_t)b0 * img_tokens(c) * c.hidden, (cudaStream_t)stream);
    if (r != DTK_OK) return r;
  }
  return DTK_OK;
}

namespace {
// copy cached positions [p0, p1) of every (layer, K|V, kv head) segment from slot src to slot dst
int copy_kv_range(dtk_engine* eng, int src, int dst, int p0, int p1, cudaStream_t s) {
  if (p1 <= p0) return DTK_OK;
  const dtk_config& c = eng->cfg;
  const size_t pitch = (size_t)c.max_len * 128 * sizeof(bf16);
  DTK_CK(cudaMemcpy2DAsync(kv_layer(eng, dst, 0) + (int64_t)p0 * 128, pitch, kv_layer(eng, src, 0) + (int64_t)p0 * 128, pitch,
                           (size_t)(p1 - p0) * 128 * sizeof(bf16), (size_t)c.layers * 2 * c.kv_heads, cudaMemcpyDeviceToDevice, s));
  return DTK_OK;
}
void drop_share(dtk_engine* eng, int slot) {
  const int b = eng->share_base[slot];
  if (b >= 0) {
    if (--eng->refcnt[b] == 0) eng->shared_upto[b] = 0;
    eng->share_base[slot] = -1;
    eng->share_len[slot] = 0;
  }
}
}  // namespace

int dtk_seq_alloc(dtk_engine* eng, int* slot) {
  if (!eng || !slot) return DTK_ERR_INVALID;
  for (size_t i = 0; i < eng->slot_used.size(); ++i)
    if (!eng->slot_used[i]) {
      eng->slot_used[i] = 1;
      *slot = (int)i;
      return DTK_OK;
    }
  eng->err = "no free KV sequence slot";
  return DTK_ERR_NOSLOT;
}

int dtk_seq_free(dtk_engine* eng, int slot) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(slot >= 0 && slot < (int)eng->slot_used.size() && eng->slot_used[slot], "slot");
  DTK_REQUIRE(eng->refcnt[slot] == 0, "slot still lends a shared prefix to other sequences (free them first)");
  drop_share(eng, slot);
  eng->slot_used[slot] = 0;
  return DTK_OK;
}

int dtk_seq_fork(dtk_engine* eng, int src, int dst, int len, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  const dtk_config& c = eng->cfg;
  DTK_REQUIRE(src >= 0 && src < c.max_seqs && dst >= 0 && dst < c.max_seqs && src != dst, "slots");
  DTK_REQUIRE(len >= 0 && len <= c.max_len, "len");
  DTK_REQUIRE(eng->refcnt[dst] == 0, "destination lends a shared prefix to other sequences");
  DTK_CK(cudaSetDevice(eng->device));
  drop_share(eng, dst);          // the copy makes dst self-contained
  if (len == 0) return DTK_OK;
  // positions below src's shared length live in its base slot
  const int sl = eng->share_len[src] < len ? eng->share_len[src] : len;
  int r = DTK_OK;
  if (sl > 0) r = copy_kv_range(eng, eng->share_base[src], dst, 0, sl, (cudaStream_t)stream);
  if (r == DTK_OK) r = copy_kv_range(eng, src, dst, sl, len, (cudaStream_t)stream);
  return r;
}

int dtk_seq_share(dtk_engine* eng, int base, int dst, int len, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  const dtk_config& c = eng->cfg;
  DTK_REQUIRE(base >= 0 && base < c.max_seqs && dst >= 0 && dst < c.max_seqs && base != dst, "slots");
  DTK_REQUIRE(eng->slot_used[base] && eng->slot_used[dst], "slots must be allocated");
  DTK_REQUIRE(len >= 0 && len <= c.max_len, "len");
  DTK_REQUIRE(eng->refcnt[dst] == 0, "destination lends a shared prefix to other sequences");
  DTK_CK(cudaSetDevice(eng->device));
  drop_share(eng, dst);
  if (len == 0) return DTK_OK;
  // one level only: if `base` itself borrows [0, L0) from a root slot, dst borrows that part from the root too
  int root = base, rootlen = len;
  if (eng->share_base[base] >= 0) {
    root = eng->share_base[base];
    rootlen = len < eng->share_len[base] ? len : eng->share_len[base];
  }
  const int s16 = rootlen & ~15;               // the decode kernel streams the cache in 16-position items
  if (s16 > 0) {
    eng->share_base[dst] = root;
    eng->share_len[dst] = s16;
    ++eng->refcnt[root];
    if (eng->shared_upto[root] < s16) eng->shared_upto[root] = s16;
  }
  // the remainder [s16, len) becomes dst's own copy: from the root up to rootlen, from base beyond
  int r = copy_kv_range(eng, root, dst, s16, rootlen, (cudaStream_t)stream);
  if (r == DTK_OK && root != base) r = copy_kv_range(eng, base, dst, rootlen, len, (cudaStream_t)stream);
  return r;
}

int dtk_prefill(dtk_engine* eng, int slot, const int64_t* ids, int T, int start_pos, const float* img_embeds,
                int img_start, int n_img, float* last_logits, float* all_logits, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  const dtk_config& c = eng->cfg;
  DTK_REQUIRE(ids && T > 0, "ids/T");
  DTK_REQUIRE(slot >= 0 && slot < c.max_seqs, "slot");
  DTK_REQUIRE(start_pos >= 0 && start_pos + T <= c.max_len, "start_pos + T exceeds max_len");
  DTK_REQUIRE(start_pos >= eng->share_len[slot], "start_pos lies inside the sequence's shared (read-only) prefix");
  DTK_REQUIRE(start_pos >= eng->shared_upto[slot], "start_pos lies inside a prefix other sequences share from this slot");
  DTK_CK(cudaSetDevice(eng->device));
  cudaStream_t s = (cudaStream_t)stream;
  uint64_t* lc = &eng->launches;
  const int H = c.hidden, I = c.inter, qd = c.heads * 128, kd = c.kv_heads * 128;
  DTK_CK(launch_embed_splice(ids, T, start_pos, W(eng, "dec.embed"), H, c.vocab, c.image_token_id, img_embeds, img_start,
                             n_img, eng->p_x, s, lc));
  for (int l = 0; l < c.layers; ++l) {
    DTK_CK(launch_rmsnorm(eng->p_x, H, W(eng, LN("dec.L", l, "norm1")), c.rms_eps, T, H, eng->p_xn, s, lc));
    {
      GemmArgs g{};
      g.A = eng->p_xn; g.lda = H; g.W = W(eng, LN("dec.L", l, "wqkv")); g.ldw = H; g.M = T; g.N = qd + 2 * kd; g.K = H;
      g.out_f32 = eng->p_qkv; g.ldo = qd + 2 * kd;
      DTK_CK(launch_gemm(g, s, lc));
    }
    bf16* kc = kv_layer(eng, slot, l);
    bf16* vc = kc + eng->kv_v_offset;
    DTK_CK(launch_rope_kv_prefill(eng->p_qkv, T, start_pos, c.heads, c.kv_heads, eng->rope_cs, eng->p_q, kc, vc, c.max_len, s, lc));
    {
      AttnArgs a{};
      a.q = eng->p_q; a.k = kc; a.v = vc; a.o = eng->p_att;
      a.q_bs = 0; a.q_hs = 128; a.q_rs = qd;
      a.k_bs = 0; a.k_hs = (int64_t)c.max_len * 128; a.k_rs = 128;
      a.v_bs = 0; a.v_hs = (int64_t)c.max_len * 128; a.v_rs = 128;
      a.o_bs = 0; a.o_hs = 128; a.o_rs = qd;
      a.B = 1; a.heads = c.heads; a.kv_group = c.heads / c.kv_heads; a.Tq = T; a.Tk = start_pos + T; a.q_pos0 = start_pos;
      a.causal = 1; a.head_dim = 128; a.scale = 1.0f / sqrtf(128.f);
      if (eng->share_len[slot] > 0) {   // keys below the shared length come from the base slot
        a.k2 = kv_layer(eng, eng->share_base[slot], l);
        a.v2 = a.k2 + eng->kv_v_offset;
        a.split_row = eng->share_len[slot];
      }
      DTK_CK(launch_flash_attn(a, s, lc));
    }
    {
      GemmArgs g{};
      g.A = eng->p_att; g.lda = qd; g.W = W(eng, LN("dec.L", l, "wo")); g.ldw = qd; g.M = T; g.N = H; g.K = qd;
      g.resid = eng->p_x; g.ldr = H; g.out_f32 = eng->p_x; g.ldo = H;
      DTK_CK(launch_gemm(g, s, lc));
    }
    DTK_CK(launch_rmsnorm(eng->p_x, H, W(eng, LN("dec.L", l, "norm2")), c.rms_eps, T, H, eng->p_xn, s, lc));
    {
      GemmArgs g{};
      g.A = eng->p_xn; g.lda = H; g.W = W(eng, LN("dec.L", l, "wgu")); g.ldw = H; g.M = T; g.N = 2 * I; g.K = H;
      g.glu = 1; g.out_bf16 = eng->p_h; g.ldo = I;
      DTK_CK(launch_gemm(g, s, lc));
    }
    {
      GemmArgs g{};
      g.A = eng->p_h; g.lda = I; g.W = W(eng, LN("dec.L", l, "wd")); g.ldw = I; g.M = T; g.N = H; g.K = I;
      g.resid = eng->p_x; g.ldr = H; g.out_f32 = eng->p_x; g.ldo = H;
      DTK_CK(launch_gemm(g, s, lc));
    }
  }
  if (last_logits) {  // final RMSNorm + lm_head on the last row only (reference computes all T rows, v1/modeling:251-257)
    GemvArgs g{};
    g.mode = GEMV_STORE; g.W = W(eng, "dec.lm_head"); g.N = c.vocab; g.K = H;
    g.x = eng->p_x + (int64_t)(T - 1) * H; g.x_stride = H; g.norm_w = W(eng, "dec.norm"); g.eps = c.rms_eps;
    g.out = last_logits; g.out_stride = c.vocab; g.B = 1;
    DTK_CK(launch_gemv(g, s, lc));
  }
  if (all_logits) {
    DTK_CK(launch_rmsnorm(eng->p_x, H, W(eng, "dec.norm"), c.rms_eps, T, H, eng->p_xn, s, lc));
    GemmArgs g{};
    g.A = eng->p_xn; g.lda = H; g.W = W(eng, "dec.lm_head"); g.ldw = H; g.M = T; g.N = c.vocab; g.K = H;
    g.out_f32 = all_logits; g.ldo = c.vocab;
    DTK_CK(launch_gemm(g, s, lc));
  }
  return DTK_OK;
}

int dtk_decode(dtk_engine* eng, const int* slots, const int* positions, const int64_t* ids, int B, float* logits,
               void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  const dtk_config& c = eng->cfg;
  DTK_REQUIRE(slots && positions && ids && logits, "null pointer");
  DTK_REQUIRE(B > 0 && B <= c.max_batch, "B exceeds max_batch");
  StateArgs st{};
  st.n = B;
  for (int i = 0; i < B; ++i) {
    DTK_REQUIRE(slots[i] >= 0 && slots[i] < c.max_seqs, "slot");
    DTK_REQUIRE(positions[i] >= 0 && positions[i] < c.max_len, "position exceeds max_len");
    DTK_REQUIRE(positions[i] >= eng->share_len[slots[i]], "position lies inside the sequence's shared (read-only) prefix");
    DTK_REQUIRE(positions[i] >= eng->shared_upto[slots[i]], "position lies inside a prefix other sequences share from this slot");
    st.slots[i] = slots[i];
    st.pos[i] = positions[i];
    st.share_slot[i] = eng->share_base[slots[i]] >= 0 ? eng->share_base[slots[i]] : slots[i];
    st.share_len[i] = eng->share_len[slots[i]];
  }
  DTK_CK(cudaSetDevice(eng->device));
  cudaStream_t s = (cudaStream_t)stream;
  set_state_kernel<<<1, 64, 0, s>>>(st, eng->d_slots, eng->d_pos, eng->d_tok, eng->d_share_slot, eng->d_share_len);
  ++eng->launches;
  DTK_CK(cudaGetLastError());
  set_cascade(eng, st);
  return decode_launches(eng, B, ids, logits, s);
}

int dtk_sample(dtk_engine* eng, const float* logits, int B, const dtk_sampling* params, const int* suppress,
               const uint32_t* steps, const uint32_t* seq_ids, int64_t* out_ids, float* probs_out, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(logits && params && B > 0 && B <= eng->cfg.max_batch, "logits/params/B");
  DTK_CK(cudaSetDevice(eng->device));
  SampleArgs a;
  fill_sample_args(eng, a, logits, B, *params);
  if (probs_out) { a.scratch = probs_out; a.want_probs = 1; }
  a.out_ids = out_ids;
  for (int i = 0; i < B; ++i) {
    a.seq[i].suppress = suppress ? suppress[i] : 0;
    a.seq[i].step = steps ? steps[i] : 0;
    a.seq[i].seq_id = seq_ids ? seq_ids[i] : (uint32_t)i;
  }
  DTK_CK(launch_sample(a, (cudaStream_t)stream, &eng->launches));
  return DTK_OK;
}

int dtk_gen_begin(dtk_engine* eng, const int* slots, const int* positions, const int64_t* first_ids_host, int B,
                  const dtk_sampling* params, const uint32_t* seq_ids, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  const dtk_config& c = eng->cfg;
  DTK_REQUIRE(slots && positions && first_ids_host && params, "null pointer");
  DTK_REQUIRE(B > 0 && B <= c.max_batch, "B exceeds max_batch");
  DTK_CK(cudaSetDevice(eng->device));
  cudaStream_t s = (cudaStream_t)stream;
  StateArgs st{};
  st.n = B; st.have_tok = 1;
  for (int i = 0; i < B; ++i) {
    DTK_REQUIRE(slots[i] >= 0 && slots[i] < c.max_seqs, "slot");
    DTK_REQUIRE(positions[i] >= 0 && positions[i] < c.max_len, "position exceeds max_len");
    DTK_REQUIRE(positions[i] >= eng->share_len[slots[i]] && positions[i] >= eng->shared_upto[slots[i]], "position lies inside a shared prefix");
    st.slots[i] = slots[i]; st.pos[i] = positions[i]; st.tok[i] = first_ids_host[i];
    st.share_slot[i] = eng->share_base[slots[i]] >= 0 ? eng->share_base[slots[i]] : slots[i];
    st.share_len[i] = eng->share_len[slots[i]];
  }
  set_cascade(eng, st);
  set_state_kernel<<<1, 64, 0, s>>>(st, eng->d_slots, eng->d_pos, eng->d_tok, eng->d_share_slot, eng->d_share_len);
  reset_gen_kernel<<<1, 1, 0, s>>>(eng->d_gen, eng->d_counters + (int64_t)c.max_batch * c.heads, params->seed);
  eng->launches += 2;
  DTK_CK(cudaGetLastError());
  DTK_CK(cudaStreamSynchronize(s));
  std::memset(eng->host_ring, 0, (size_t)eng->ring * 64 * sizeof(unsigned long long));  // stamps restart at step 1

  eng->gen_B = B;
  eng->gen_params = *params;
  eng->gen_stream = s;
  {  // sampler arguments of the loop (suppress = 0, RNG counter = 1 + step)
    SampleArgs& a = eng->gen_sample;
    fill_sample_args(eng, a, eng->d_logits, B, *params);
    for (int i = 0; i < B; ++i) { a.seq[i].suppress = 0; a.seq[i].step = 1; a.seq[i].seq_id = seq_ids ? seq_ids[i] : (uint32_t)i; }
    a.gen_tok = eng->d_tok; a.gen_pos = eng->d_pos; a.gen_step = eng->d_gen; a.seed_dev = eng->d_gen + 1; a.seed = 0;
    a.host_ring = eng->dev_ring; a.ring = eng->ring;
    a.done_counter = eng->d_counters + (int64_t)c.max_batch * c.heads;
  }
  eng->gen_mega = (B == 1 && eng->decode_impl == 1 && eng->mega_ok);
  eng->gen_fused = eng->gen_mega && eng->fuse_greedy && !eng->gen_sample.do_sample;
  if (eng->gen_mega) {  // one cooperative launch (+ sampler when sampling) per token: no graph needed
    eng->gen_graph = nullptr;
    return DTK_OK;
  }
  // graph key: everything baked into kernel arguments
  char key[256];
  std::snprintf(key, sizeof(key), "B%d|t%.9g|p%.17g|k%d|s%d|b%d|e%d", B, (double)params->temperature,
                (double)params->top_p, params->top_k, params->do_sample, params->bad_token, params->begin_suppress_token);
  std::string skey(key);
  skey += "|g" + std::to_string(eng->decode_gemm_min_batch) + "|i" + std::to_string(get_gemm_impl());
  skey += "|c" + std::to_string(eng->cas_slot) + ":" + std::to_string(eng->cas_len);   // shared-prefix attention bakes slot and length in
  if (seq_ids) for (int i = 0; i < B; ++i) skey += "," + std::to_string(seq_ids[i]);
  auto it = eng->graphs.find(skey);
  if (it == eng->graphs.end()) {
    cudaGraph_t graph = nullptr;
    uint64_t before = eng->launches;
    if (!eng->cap_stream) DTK_CK(cudaStreamCreateWithFlags(&eng->cap_stream, cudaStreamNonBlocking));
    cudaStream_t cs = eng->cap_stream;
    DTK_CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    int r = decode_launches(eng, B, nullptr, eng->d_logits, cs);
    if (r == DTK_OK) {
      cudaError_t e = launch_sample(eng->gen_sample, cs, &eng->launches);
      if (e != cudaSuccess) { eng->err = std::string("launch_sample: ") + cudaGetErrorString(e); r = DTK_ERR_CUDA; }
    }
    cudaError_t ce = cudaStreamEndCapture(cs, &graph);
    eng->launches = before;  // captured launches are counted per replay
    if (r != DTK_OK) { if (graph) cudaGraphDestroy(graph); return r; }
    if (ce != cudaSuccess) { eng->err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce); return DTK_ERR_CUDA; }
    cudaGraphExec_t exec = nullptr;
    DTK_CK(cudaGraphInstantiate(&exec, graph, 0));
    cudaGraphDestroy(graph);
    if (eng->graphs.size() >= 64) {  // bound the cache
      for (auto& g : eng->graphs) cudaGraphExecDestroy(g.second);
      eng->graphs.clear();
    }
    it = eng->graphs.emplace(skey, exec).first;
  }
  eng->gen_graph = it->second;
  return DTK_OK;
}

int dtk_gen_step(dtk_engine* eng, void* stream) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(eng->gen_B > 0, "dtk_gen_begin not called");
  if (eng->gen_mega) {
    int r = decode_launches(eng, 1, nullptr, eng->d_logits, (cudaStream_t)stream);
    if (r != DTK_OK) return r;
    if (!eng->gen_fused) DTK_CK(launch_sample(eng->gen_sample, (cudaStream_t)stream, &eng->launches));
    return DTK_OK;
  }
  DTK_REQUIRE(eng->gen_graph != nullptr, "dtk_gen_begin not called");
  DTK_CK(cudaGraphLaunch(eng->gen_graph, (cudaStream_t)stream));
  const bool gemm_path = eng->decode_gemm_min_batch > 0 && eng->gen_B >= eng->decode_gemm_min_batch;
  eng->launches += gemm_path ? (uint64_t)eng->cfg.layers * (9 + (eng->cas_len > 0 ? 1 : 0)) + 4 : (uint64_t)eng->cfg.layers * 5 + 3;   // kernels per replay
  return DTK_OK;
}

int dtk_gen_wait(dtk_engine* eng, int64_t step, int32_t* tokens_out_host) {
  if (!eng) return DTK_ERR_INVALID;
  DTK_REQUIRE(eng->gen_B > 0 && step >= 0 && tokens_out_host, "gen state/step/out");
  // every sequence's entry of this step carries the stamp step + 1 in its upper half (one 8-byte device store)
  volatile const unsigned long long* row = eng->host_ring + (size_t)(step % eng->ring) * eng->gen_B;
  const unsigned long long want = (unsigned long long)(step + 1);
  auto t0 = std::chrono::steady_clock::now();
  uint64_t spins = 0;
  for (int i = 0; i < eng->gen_B; ++i) {
    unsigned long long e;
    while (((e = row[i]) >> 32) != want) {
      if ((e >> 32) > want) {   // the device is a whole ring ahead: the token was overwritten
        eng->err = "token ring overrun: dtk_gen_wait lagged more than the ring depth behind dtk_gen_step";
        return DTK_ERR_INVALID;
      }
      if ((++spins & 0x3ff) == 0) {
        cudaError_t q = cudaStreamQuery(eng->gen_stream);
        if (q != cudaSuccess && q != cudaErrorNotReady) {
          eng->err = std::string("stream error while waiting for token: ") + cudaGetErrorString(q);
          return DTK_ERR_CUDA;
        }
        if (q == cudaSuccess && (row[i] >> 32) != want) {
          eng->err = "stream idle but requested step was never launched";
          return DTK_ERR_INVALID;
        }
        if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(60)) {
          eng->err = "timeout waiting for generated token";
          return DTK_ERR_CUDA;
        }
      }
    }
    tokens_out_host[i] = (int32_t)(uint32_t)(e & 0xffffffffull);
  }
  return DTK_OK;
}

int dtk_gen_end(dtk_engine* eng) {
  if (!eng) return DTK_ERR_INVALID;
  if (eng->gen_B > 0) {
    DTK_CK(cudaSetDevice(eng->device));
    DTK_CK(cudaStreamSynchronize(eng->gen_stream));
  }
  eng->gen_graph = nullptr;
  eng->gen_mega = false;
  eng->gen_fused = false;
  eng->gen_B = 0;
  return DTK_OK;
}

int dtk_set_option(dtk_engine* eng, const char* key, int64_t value) {
  if (!eng || !key) return DTK_ERR_INVALID;
  DTK_REQUIRE(eng->gen_B == 0, "options cannot change inside a generation loop");
  if (std::strcmp(key, "decode_impl") == 0) {
    DTK_REQUIRE(value == 0 || value == 1, "decode_impl must be 0 (per-op) or 1 (persistent)");
    eng->decode_impl = (int)value;
    return DTK_OK;
  }
  if (std::strcmp(key, "decode_gemm_min_batch") == 0) {  // 0 = never; default 4
    DTK_REQUIRE(value >= 0 && value <= 64, "decode_gemm_min_batch must be in 0..64");
    eng->decode_gemm_min_batch = (int)value;
    return DTK_OK;
  }
  if (std::strcmp(key, "gemm_impl") == 0) {  // process-wide dev switch: 0 = mma.sync, 1 = tcgen05 where supported
    DTK_REQUIRE(value >= 0 && value <= 3, "gemm_impl must be 0..3");
    set_gemm_impl((int)value);
    return DTK_OK;
  }
  if (std::strcmp(key, "cascade_attn") == 0) {  // 1 (default) = shared-prefix attention for batched steps whose rows share one prefix
    eng->cascade_attn = value ? 1 : 0;
    return DTK_OK;
  }
  if (std::strcmp(key, "gemm_swap_split") == 0) {  // process-wide dev switch: split-K factor of the batched-decode GEMM
    DTK_REQUIRE(value >= 0 && value <= 8, "gemm_swap_split must be 0 (heuristic) .. 8");
    set_gemm_swap_split((int)value);
    return DTK_OK;
  }
  if (std::strcmp(key, "gemm_skinny_swap") == 0) {  // process-wide dev switch
    set_gemm_skinny_swap(value ? 1 : 0);
    return DTK_OK;
  }
  if (std::strcmp(key, "sample_impl") == 0) {  // process-wide: 0 = register-resident sampler when V fits, 1 = generic kernel
    DTK_REQUIRE(value == 0 || value == 1, "sample_impl must be 0 or 1");
    set_sample_impl((int)value);
    return DTK_OK;
  }
  if (std::strcmp(key, "mega_flags") == 0) {  // dev only (timing experiments; results are garbage when set)
    eng->mega_flags = (int)value;
    return DTK_OK;
  }
  if (std::strcmp(key, "mega_debug") == 0) {
    eng->mega_debug = value ? 1 : 0;
    return DTK_OK;
  }
  if (std::strcmp(key, "attn_impl") == 0) {  // ViT attention: 1 (default) = tcgen05, 0 = mma.sync
    DTK_REQUIRE(value == 0 || value == 1, "attn_impl must be 0 or 1");
    eng->attn_impl = (int)value;
    return DTK_OK;
  }
  if (std::strcmp(key, "fuse_greedy") == 0) {  // 1 (default): greedy generation loops take the argmax in the decode kernel's tail
    eng->fuse_greedy = value ? 1 : 0;
    return DTK_OK;
  }
  if (std::strcmp(key, "vit_graph") == 0) {  // 1 (default) = ViT chunks replayed from CUDA graphs, 0 = direct launches
    eng->vit_graph = value ? 1 : 0;
    return DTK_OK;
  }
  if (std::strcmp(key, "mega_variant") == 0) {  // dev A/B switches of the persistent kernel (results identical)
    eng->mega_variant = (int)value;
    return DTK_OK;
  }
  if (std::strcmp(key, "mega_nslots") == 0) {  // dev: smaller ring (8 / 16) for A/B runs of the stream's depth
    eng->mega_nslots = (int)value;
    return DTK_OK;
  }
  if (std::strcmp(key, "mega_trace_layer") == 0) {  // dev: per-tile clock trace of this layer (-1 = off); needs mega_debug
    eng->mega_trace_layer = (int)value;
    return DTK_OK;
  }
  eng->err = std::string("unknown option ") + key;
  return DTK_ERR_INVALID;
}

int dtk_get_option(dtk_engine* eng, const char* key, int64_t* value) {
  if (!eng || !key || !value) return DTK_ERR_INVALID;
  if (std::strcmp(key, "decode_impl") == 0) { *value = eng->decode_impl; return DTK_OK; }
  if (std::strcmp(key, "decode_persistent") == 0) { *value = (eng->decode_impl == 1 && eng->mega_ok) ? 1 : 0; return DTK_OK; }
  if (std::strcmp(key, "gemm_impl") == 0) { *value = get_gemm_impl(); return DTK_OK; }
  if (std::strcmp(key, "decode_gemm_min_batch") == 0) { *value = eng->decode_gemm_min_batch; return DTK_OK; }
  if (std::strcmp(key, "sample_impl") == 0) { *value = get_sample_impl(); return DTK_OK; }
  if (std::strcmp(key, "mega_flags") == 0) { *value = eng->mega_flags; return DTK_OK; }
  if (std::strcmp(key, "mega_debug") == 0) { *value = eng->mega_debug; return DTK_OK; }
  if (std::strcmp(key, "mega_variant") == 0) { *value = eng->mega_variant; return DTK_OK; }
  eng->err = std::string("unknown option ") + key;
  return DTK_ERR_INVALID;
}

// ---- kernel-level test hooks ---------------------------------------------------------------
int dtk_dbg_mega_times(dtk_engine* eng, long long* out_host, int max_values) {
  if (!eng || !out_host) return DTK_ERR_INVALID;
  DTK_REQUIRE(eng->d_dbg != nullptr, "persistent kernel unavailable");
  const int n = eng->mega_grid * (eng->cfg.layers * 5 + 1) * 4;
  DTK_CK(cudaSetDevice(eng->device));
  DTK_CK(cudaDeviceSynchronize());
  DTK_CK(cudaMemcpy(out_host, eng->d_dbg, (size_t)(n < max_values ? n : max_values) * sizeof(long long), cudaMemcpyDeviceToHost));
  return n;
}

int dtk_dbg_mega_trace(dtk_engine* eng, long long* out_host, int max_values) {
  if (!eng || !out_host) return DTK_ERR_INVALID;
  DTK_REQUIRE(eng->d_dbg2 != nullptr, "persistent kernel unavailable");
  const int n = eng->mega_grid * MEGA_DBG2_ROWS * 4;
  DTK_CK(cudaSetDevice(eng->device));
  DTK_CK(cudaDeviceSynchronize());
  DTK_CK(cudaMemcpy(out_host, eng->d_dbg2, (size_t)(n < max_values ? n : max_values) * sizeof(long long), cudaMemcpyDeviceToHost));
  return n;
}

int dtk_dbg_gemm_impl(int impl) {
  if (impl >= 0) {
    set_gemm_impl(impl & 0xff);
    set_gemm_swap_split((impl >> 8) & 0xf);   // forced split-K factor of the batched-decode tile (0 = heuristic)
  }
  return get_gemm_impl();
}

int dtk_dbg_gemm(const void* A, const void* Wm, const void* bias, const float* resid, int M, int N, int K, int act,
                 int glu, float* out_f32, void* out_bf16, void* stream) {
  GemmArgs g{};
  g.A = (const bf16*)A; g.lda = K; g.W = (const bf16*)Wm; g.ldw = K; g.M = M; g.N = N; g.K = K;
  g.bias = (const bf16*)bias; g.resid = resid; g.ldr = glu ? N / 2 : N; g.act = act; g.glu = glu;
  g.out_f32 = out_f32; g.out_bf16 = (bf16*)out_bf16; g.ldo = glu ? N / 2 : N;
  return launch_gemm(g, (cudaStream_t)stream, nullptr) == cudaSuccess ? DTK_OK : DTK_ERR_CUDA;
}

int dtk_dbg_flash_attn(const void* q, const void* k, const void* v, void* o, int B, int heads, int Tq, int Tk,
                       int head_dim, int causal, int q_pos0, float scale, void* stream) {
  AttnArgs a{};
  a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.o = (bf16*)o;
  const int64_t rs = (int64_t)heads * head_dim;
  a.q_bs = (int64_t)Tq * rs; a.q_hs = head_dim; a.q_rs = rs;
  a.k_bs = (int64_t)Tk * rs; a.k_hs = head_dim; a.k_rs = rs;
  a.v_bs = (int64_t)Tk * rs; a.v_hs = head_dim; a.v_rs = rs;
  a.o_bs = (int64_t)Tq * rs; a.o_hs = head_dim; a.o_rs = rs;
  a.B = B; a.heads = heads; a.kv_group = 1; a.Tq = Tq; a.Tk = Tk; a.q_pos0 = q_pos0; a.causal = causal;
  a.head_dim = head_dim; a.scale = scale;
  return launch_flash_attn(a, (cudaStream_t)stream, nullptr) == cudaSuccess ? DTK_OK : DTK_ERR_CUDA;
}

int dtk_dbg_flash_attn_ex(const void* q, const void* k, const void* v, const void* k2, const void* v2, void* o, int B,
                          int heads, int kv_heads, int Tq, int Tk, int head_dim, int causal, int q_pos0, int split_row,
                          float scale, void* stream) {
  if (!q || !k || !v || !o || B <= 0 || heads <= 0 || kv_heads <= 0 || heads % kv_heads || Tq <= 0 || Tk <= 0)
    return DTK_ERR_INVALID;
  if ((head_dim != 72 && head_dim != 128) || q_pos0 < 0 || split_row < 0 || split_row > Tk) return DTK_ERR_INVALID;
  if (split_row > 0 && (!k2 || !v2)) return DTK_ERR_INVALID;
  AttnArgs a{};
  a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.o = (bf16*)o;
  a.k2 = (const bf16*)k2; a.v2 = (const bf16*)v2; a.split_row = split_row;
  const int64_t rs = (int64_t)heads * head_dim, krs = (int64_t)kv_heads * head_dim;
  a.q_bs = (int64_t)Tq * rs; a.q_hs = head_dim; a.q_rs = rs;
  a.k_bs = (int64_t)Tk * krs; a.k_hs = head_dim; a.k_rs = krs;
  a.v_bs = (int64_t)Tk * krs; a.v_hs = head_dim; a.v_rs = krs;
  a.o_bs = (int64_t)Tq * rs; a.o_hs = head_dim; a.o_rs = rs;
  a.B = B; a.heads = heads; a.kv_group = heads / kv_heads; a.Tq = Tq; a.Tk = Tk; a.q_pos0 = q_pos0; a.causal = causal;
  a.head_dim = head_dim; a.scale = scale;
  return launch_flash_attn(a, (cudaStream_t)stream, nullptr) == cudaSuccess ? DTK_OK : DTK_ERR_CUDA;
}

int dtk_dbg_decode_attn(const float* q, const void* kv, int nslots, const int* slots, const int* pos,
                        const int* share_slot, const int* share_len, int B, int heads, int kv_heads, int max_len,
                        int nsplit, float scale, float* part_o, float* part_ml, unsigned int* counters, float* out,
                        void* out_bf16, const void* q_bf16, int prefix_slot, int prefix_len, int part_tiles,
                        void* stream) {
  if (!q || !kv || !slots || !pos || !part_o || !part_ml || !counters || !out) return DTK_ERR_INVALID;
  if (B <= 0 || B > 64 || heads <= 0 || kv_heads <= 0 || heads % kv_heads || max_len <= 0 || nslots <= 0)
    return DTK_ERR_INVALID;
  if (nsplit < 1 || nsplit > 16 || prefix_len < 0 || prefix_len > max_len) return DTK_ERR_INVALID;
  int csplit = 0;
  if (prefix_len > 0) {   // the engine's shared-prefix ("cascade") pass: launch_flash_attn in partial mode, then the merge
    if (!q_bf16 || part_tiles <= 0 || prefix_slot < 0 || prefix_slot >= nslots) return DTK_ERR_INVALID;
    csplit = ((prefix_len + 63) / 64 + part_tiles - 1) / part_tiles;
    if (nsplit + csplit > 16) return DTK_ERR_INVALID;   // partial buffers hold 16 slots per (row, head)
  }
  // the per-row state lives on the device: check it on the host so that no launch indexes outside the KV buffer
  std::vector<int> h_slots(B), h_pos(B), h_sslot(B, 0), h_slen(B, 0);
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaStreamSynchronize(s) != cudaSuccess) return DTK_ERR_CUDA;
  bool ok = cudaMemcpy(h_slots.data(), slots, B * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess &&
            cudaMemcpy(h_pos.data(), pos, B * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess;
  if (ok && share_len) {
    if (!share_slot) return DTK_ERR_INVALID;
    ok = cudaMemcpy(h_sslot.data(), share_slot, B * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess &&
         cudaMemcpy(h_slen.data(), share_len, B * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess;
  }
  if (!ok) return DTK_ERR_CUDA;
  for (int b = 0; b < B; ++b) {
    if (h_slots[b] < 0 || h_slots[b] >= nslots || h_pos[b] < prefix_len || h_pos[b] >= max_len) return DTK_ERR_INVALID;
    if (h_slen[b] < 0 || h_slen[b] > max_len) return DTK_ERR_INVALID;
    if (h_slen[b] > 0 && (h_sslot[b] < 0 || h_sslot[b] >= nslots)) return DTK_ERR_INVALID;
  }
  // one layer of the engine's slot-major cache: [slot][K | V][kv_head][max_len][128]
  const int64_t v_off = (int64_t)kv_heads * max_len * 128;
  const bf16* kvb = (const bf16*)kv;
  if (prefix_len > 0) {
    AttnArgs f{};
    f.q = (const bf16*)q_bf16; f.k = kvb + prefix_slot * 2 * v_off; f.v = f.k + v_off;
    f.q_bs = 0; f.q_hs = 128; f.q_rs = (int64_t)heads * 128;
    f.k_bs = 0; f.k_hs = (int64_t)max_len * 128; f.k_rs = 128;
    f.v_bs = 0; f.v_hs = (int64_t)max_len * 128; f.v_rs = 128;
    f.B = 1; f.heads = heads; f.kv_group = heads / kv_heads; f.Tq = B; f.Tk = prefix_len; f.q_pos0 = 0;
    f.causal = 0; f.head_dim = 128; f.scale = scale;
    f.part_o = part_o; f.part_ml = part_ml; f.part_np = nsplit + csplit; f.part_idx0 = nsplit; f.part_tiles = part_tiles;
    if (launch_flash_attn(f, s, nullptr) != cudaSuccess) return DTK_ERR_CUDA;
  }
  DecodeAttnArgs a{};
  a.q = q; a.q_stride = (int64_t)heads * 128; a.kv_base = kvb; a.kv_slot_stride = 2 * v_off; a.kv_v_offset = v_off;
  a.slots = slots; a.pos = pos; a.share_slot = share_slot; a.share_len = share_len;
  a.B = B; a.heads = heads; a.kv_group = heads / kv_heads; a.max_len = max_len; a.nsplit = nsplit; a.scale = scale;
  a.part_o = part_o; a.part_ml = part_ml; a.counters = counters;
  a.out = out; a.out_stride = (int64_t)heads * 128; a.out_bf16 = (bf16*)out_bf16;
  if (prefix_len > 0) { a.key_begin = prefix_len; a.np = nsplit + csplit; }
  return launch_decode_attn(a, s, nullptr) == cudaSuccess ? DTK_OK : DTK_ERR_CUDA;
}

int dtk_dbg_attn_tc(const void* qkv, void* vt_scratch, void* o, int B, int heads, int N, float scale, void* stream) {
  if (!qkv || !vt_scratch || !o || B <= 0 || heads <= 0 || N <= 0) return DTK_ERR_INVALID;
  if (!attn_tc_supported()) return DTK_ERR_UNSUPPORTED;
  return launch_attn_tc((const bf16*)qkv, (bf16*)vt_scratch, (bf16*)o, B, heads, N, scale, (cudaStream_t)stream, nullptr) == cudaSuccess ? DTK_OK : DTK_ERR_CUDA;
}

int dtk_dbg_gemv(const void* Wm, const float* x, const void* norm_w, float eps, int N, int K, int mode, float* out,
                 void* stream) {
  if (mode < 0 || mode > 2) return DTK_ERR_INVALID;
  GemvArgs g{};
  g.mode = mode; g.W = (const bf16*)Wm; g.N = N; g.K = K; g.x = x; g.x_stride = K; g.norm_w = (const bf16*)norm_w;
  g.eps = eps; g.out = out; g.out_stride = N; g.B = 1;
  return launch_gemv(g, (cudaStream_t)stream, nullptr) == cudaSuccess ? DTK_OK : DTK_ERR_CUDA;
}

}  // extern "C"
