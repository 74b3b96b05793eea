/*
 * detikzify_b200 — C ABI of the B200-native engine for DeTikZify's image-conditioned
 * autoregressive hot path (SigLIP ViT encode -> concat-3 projector -> LLaMA prefill +
 * KV-cached decode + sampler).
 *
 * The reference (potamides/DeTikZify) is pure Python and has no FFI layer; the seam is the
 * duck-typed HF model object returned by detikzify.model.load() (detikzify/model/__init__.py:28).
 * This header is the boundary inserted *below* that seam (SURVEY.md §8b): every entry point
 * names the reference code it replaces. Conventions:
 *   - every call returns int: 0 = ok, <0 = dtk_status error; no exceptions / abort() cross
 *     the boundary; dtk_last_error() gives the message of the last failing call on that engine;
 *   - all tensor pointers are BORROWED device pointers (row-major, dense) that the caller keeps
 *     alive until the stream has consumed them; the engine owns only KV slots + workspace;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no global state; one engine per device; calls on one engine must be serialised by the
 *     caller, distinct engines are independent (the 8-GPU figure-sharded case).
 */
#ifndef DETIKZIFY_B200_H
#define DETIKZIFY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTK_ABI_VERSION 2

#if defined(__GNUC__)
#define DTK_API __attribute__((visibility("default")))
#else
#define DTK_API
#endif

typedef enum dtk_status {
  DTK_OK = 0,
  DTK_ERR_INVALID = -1,   /* bad argument / shape / state */
  DTK_ERR_CUDA = -2,      /* CUDA runtime error (message in dtk_last_error) */
  DTK_ERR_OOM = -3,       /* device allocation failed */
  DTK_ERR_NOSLOT = -4,    /* no free KV sequence slot */
  DTK_ERR_UNSUPPORTED = -5
} dtk_status;

/* Model shape. Mirrors LlamaConfig / timm-SigLIP dims the reference loads
 * (detikzify/model/v1/configuration_detikzify.py:3-13, SURVEY.md Appendix A). */
typedef struct dtk_config {
  /* decoder */
  int32_t hidden, inter, layers, heads, kv_heads, head_dim, vocab, max_len;
  float rms_eps, rope_theta, rope_factor;
  /* RoPE frequency scaling: 0 = linear (inv_freq / rope_factor; DeepSeek-Coder decoders of the v1 checkpoints),
   * 1 = "llama3" (HF modeling_rope_utils._compute_llama3_parameters; LLaMA-3.x decoders of the v2 checkpoints,
   * detikzify/model/configuration_detikzify.py:83-120): wavelengths above rope_orig_max_pos / rope_low_freq are divided by
   * rope_factor, those below rope_orig_max_pos / rope_high_freq are kept, the band in between is interpolated */
  int32_t rope_type;
  float rope_low_freq, rope_high_freq;
  int32_t rope_orig_max_pos;
  /* vision tower */
  int32_t v_hidden, v_inter, v_layers, v_heads, v_image, v_patch;
  int32_t v_act;              /* 0 = gelu_pytorch_tanh, 1 = exact (erf) gelu */
  float v_eps;
  /* glue */
  int32_t concat;             /* patches concatenated per image token (3) */
  int32_t image_token_id, eos_token_id;
  /* engine sizing */
  int32_t max_seqs;           /* KV sequence slots (each max_len positions) */
  int32_t max_batch;          /* max concurrently decoded sequences */
} dtk_config;

typedef struct dtk_weight_info {
  char name[64];
  uint64_t offset;            /* byte offset in the arena (256-B aligned) */
  uint64_t nbytes;
  int32_t rows, cols;         /* bf16 [rows, cols] row-major (cols = 1-D length if rows==1) */
} dtk_weight_info;

/* Sampling controls == the kwargs detikzify/infer/generate.py:218-227,379-387 passes to HF
 * generate (temperature/top_p/top_k/do_sample + bad_words_ids=[[image_token]] +
 * begin_suppress_tokens=[eos]). */
typedef struct dtk_sampling {
  double temperature;         /* < 1e-5 or do_sample==0 -> greedy argmax */
  double top_p;               /* >= 1 -> off (double: HF compares against python 1 - top_p) */
  int32_t top_k;              /* 0 -> off */
  int32_t do_sample;
  int32_t bad_token;          /* always masked (-1 = none) */
  int32_t begin_suppress_token; /* masked when suppress flag set (-1 = none) */
  uint64_t seed;
} dtk_sampling;

typedef struct dtk_engine dtk_engine;

DTK_API int dtk_abi_version(void);

/* ---- weights: one contiguous bf16 arena (single ncclBroadcast at load, SURVEY.md §8e) ---- */
DTK_API int dtk_weight_count(const dtk_config* cfg);
DTK_API int dtk_weight_get(const dtk_config* cfg, int index, dtk_weight_info* out);
DTK_API uint64_t dtk_arena_bytes(const dtk_config* cfg);

/* ---- lifecycle. Replaces DetikzifyForCausalLM.from_pretrained + initialize_vision_modules
 *      (detikzify/model/v1/__init__.py:24-56, v1/modeling_detikzify.py:84-117). ------------ */
DTK_API int dtk_create(const dtk_config* cfg, const void* weight_arena, uint64_t arena_bytes,
               int device, dtk_engine** out);
DTK_API int dtk_destroy(dtk_engine* eng);
DTK_API const char* dtk_last_error(const dtk_engine* eng);

/* ---- ViT. Replaces DetikzifyVisionModel.forward / get_intermediate_layers
 *      (v1/modeling_detikzify.py:63-72) == timm forward_features (+ forward_head).
 *      pixels fp32 [B,3,S,S]; tokens_out fp32 [B,N,D] (may be NULL); pooled_out fp32 [B,D]
 *      (may be NULL; attention-pool head, used by SelfSim evaluate/imagesim.py:101-103). ---- */
DTK_API int dtk_vit_encode(dtk_engine* eng, const float* pixels, int B, float* tokens_out,
                   float* pooled_out, void* stream);

/* ---- image preprocessing on the device. Replaces DetikzifyImageProcessor.preprocess for images already uploaded as
 *      uint8 (detikzify/model/v1/processing_detikzify.py:242-251: bicubic resize to SxS, x 1/255, (x - mean) / std, CHW).
 *      rgb: device uint8 [h, w, 3]; the resize is Pillow's 8-bit resampler bit for bit: bounds_* int32 [S][2] = {first
 *      input index, tap count}, coef_* int32 [S][ksize_*] = 22-bit fixed-point taps for the horizontal / vertical pass
 *      (host-computed from (w -> S) and (h -> S), see model/processing.py::pil_resample_coeffs); tmp: device uint8
 *      [h, S, 3] scratch; out: device fp32 [3, S, S]; out_u8 (may be NULL): the resized uint8 image [S, S, 3] (tests). ---- */
DTK_API int dtk_image_preprocess(dtk_engine* eng, const uint8_t* rgb, int h, int w, int S,
                                 const int32_t* bounds_h, const int32_t* coef_h, int ksize_h,
                                 const int32_t* bounds_v, const int32_t* coef_v, int ksize_v,
                                 float rescale, const float* mean3_host, const float* std3_host,
                                 uint8_t* tmp, float* out, uint8_t* out_u8, void* stream);

/* ---- concat-3 + mm_projector (v1/modeling_detikzify.py:132-137,163).
 *      tokens fp32 [B,N,D] -> out fp32 [B,P,H]; the reshape is folded into addressing. ------ */
DTK_API int dtk_project(dtk_engine* eng, const float* tokens, int B, float* out, void* stream);

/* ---- KV sequence slots (replaces DynamicCache, HF cache_utils; SURVEY.md §8f.1). ---------- */
DTK_API int dtk_seq_alloc(dtk_engine* eng, int* slot);
DTK_API int dtk_seq_free(dtk_engine* eng, int slot);
/* copy the first `len` cached positions of src into dst (dst becomes self-contained) */
DTK_API int dtk_seq_fork(dtk_engine* eng, int src_slot, int dst_slot, int len, void* stream);
/* make dst READ the first `len` cached positions from base instead of holding a copy (MCTS rollouts of one figure share the
 * image prefix and the tree path: detikzify/infer/generate.py:246-257,305-313 re-prefills them per rollout). The shared
 * part is reference counted: base cannot be freed, nor rewritten below the shared length, while a borrower exists; dst
 * writes only positions >= len. Whole 16-position blocks are shared, the remainder (< 16 positions) is copied into dst.
 * One level: sharing from a slot that itself borrows resolves to the root slot. */
DTK_API int dtk_seq_share(dtk_engine* eng, int base_slot, int dst_slot, int len, void* stream);

/* ---- prefill. Replaces DetikzifyModel.forward splice + LlamaModel.forward + lm_head for a
 *      prompt (v1/modeling_detikzify.py:144-200,218-257). Processes ids[0..T) as positions
 *      [start_pos, start_pos+T) of `slot` (positions < start_pos must already be cached).
 *      Rows whose id == image_token_id take their embedding from img_embeds (fp32 [P,H],
 *      row = position - img_start) — the count/contiguity validation is the caller's
 *      (Python shim) job. Writes fp32 logits of the LAST position to last_logits [V]
 *      (may be NULL). all_logits (may be NULL): fp32 [T,V] for parity tests. --------------- */
DTK_API int dtk_prefill(dtk_engine* eng, int slot, const int64_t* ids, int T, int start_pos,
                const float* img_embeds, int img_start, int n_img,
                float* last_logits, float* all_logits, void* stream);

/* ---- single-token decode for B sequences (LlamaModel.forward with cache, q_len == 1;
 *      v1/modeling_detikzify.py:285-305). slots: host int[B]; positions host int[B] (the
 *      position the token occupies); ids: device int64[B]; logits: device fp32 [B,V]. ------ */
DTK_API int dtk_decode(dtk_engine* eng, const int* slots, const int* positions, const int64_t* ids,
               int B, float* logits, void* stream);

/* ---- sampler. Replaces HF LogitsProcessorList + softmax + multinomial / argmax
 *      (HF generation/utils.py:2762-2793). logits fp32 [B,V]; suppress: host int[B]
 *      (1 = apply begin_suppress_token, i.e. first new token); steps: host uint32[B] RNG
 *      counters; out_ids device int64[B]; probs_out (may be NULL) fp32 [B,V] receives the
 *      post-processor probability vector (parity tests). ----------------------------------- */
DTK_API int dtk_sample(dtk_engine* eng, const float* logits, int B, const dtk_sampling* params,
               const int* suppress, const uint32_t* steps, const uint32_t* seq_ids,
               int64_t* out_ids, float* probs_out, void* stream);

/* ---- fused generation loop state (device-resident; one graph launch per token).
 *      dtk_gen_begin: bind B slots whose prompts are prefilled to `positions[b]` tokens and
 *      whose first pending token is first_ids[b] (already sampled from the prefill logits).
 *      dtk_gen_step: decode + sample one token for every bound sequence; token b of step s is
 *      written to host_ring (pinned, int32 [ring][B]) at row s % ring. Returns immediately
 *      (asynchronous on `stream`). dtk_gen_wait blocks until step s has landed. ------------- */
DTK_API int dtk_gen_begin(dtk_engine* eng, const int* slots, const int* positions,
                  const int64_t* first_ids_host, int B, const dtk_sampling* params,
                  const uint32_t* seq_ids, void* stream);
DTK_API int dtk_gen_step(dtk_engine* eng, void* stream);
DTK_API int dtk_gen_wait(dtk_engine* eng, int64_t step, int32_t* tokens_out_host /* [B] */);
DTK_API int dtk_gen_end(dtk_engine* eng);

/* ---- engine options. "decode_impl": 1 = persistent weight-streaming decode kernel (default for
 *      B = 1), 0 = per-op kernels replayed from a CUDA graph (always used for B > 1). Others (all with
 *      working defaults): "gemm_impl" (see dtk_dbg_gemm_impl), "attn_impl" (ViT attention: 1 = tcgen05, 0 =
 *      mma.sync), "cascade_attn" (shared-prefix attention of batched decode), "decode_gemm_min_batch",
 *      "fuse_greedy", "vit_graph", and dev switches "mega_debug", "mega_flags", "mega_trace_layer",
 *      "mega_nslots", "mega_variant". Unknown keys return DTK_ERR_INVALID. ------------------------- */
DTK_API int dtk_set_option(dtk_engine* eng, const char* key, int64_t value);
/*      Read back an option; the extra key "decode_persistent" reports whether B = 1 decode steps
 *      actually run on the persistent kernel (option set AND the device can co-schedule its grid). */
DTK_API int dtk_get_option(dtk_engine* eng, const char* key, int64_t* value);

/* ---- introspection for benches: algorithmic HBM bytes of one decode step at context T ----- */
DTK_API uint64_t dtk_decode_bytes(const dtk_config* cfg, int context_len);
/* kernels launched by this engine since creation (bench.py's gpu_launches) */
DTK_API uint64_t dtk_launch_count(const dtk_engine* eng);

/* ---- kernel-level test hooks (used only by tests/: shape sweeps at the real model sizes
 *      without instantiating a model). All pointers are device pointers. --------------------- */
/* phase timestamps of the last persistent-kernel launch (option "mega_debug" = 1):
 * [grid CTAs][5*layers+1 phases][4] globaltimer (ns) stamps; returns the value count */
DTK_API int dtk_dbg_mega_times(dtk_engine* eng, long long* out_host, int max_values);
/* per-tile SM-clock trace of one layer (options "mega_debug" = 1, "mega_trace_layer" = l): [grid CTAs][168 rows][4];
 * rows 0..159 = the CTA's local tiles of that layer {producer issue, bytes landed, tile done, consumer asked},
 * rows 160..164 = the layer's five phases {start, staged, items done, barrier done}; returns the value count */
DTK_API int dtk_dbg_mega_trace(dtk_engine* eng, long long* out_host, int max_values);
/* select the dense GEMM implementation used by dtk_dbg_gemm and the engines of this process:
 * 0 = mma.sync, 1 = tcgen05 one 128 x 128 tile per CTA, 2 (default) = persistent 128 x 256 tcgen05 kernel with two TMEM
 * accumulators, 3 = CTA-pair (cta_group::2) 256 x 256 kernel, -1 = query only; returns the current setting. Bits 8..11 of a
 * non-negative value force the split-K factor (cluster size 1..8) of the batched-decode tile; 0 = heuristic. */
DTK_API int dtk_dbg_gemm_impl(int impl);
/* C = act(A[M,K] * W[N,K]^T + bias) (+resid); glu: out[m, n/2] = silu(c[m,n]) * c[m,n+1] */
DTK_API int dtk_dbg_gemm(const void* A_bf16, const void* W_bf16, const void* bias_bf16,
                         const float* resid, int M, int N, int K, int act, int glu,
                         float* out_f32, void* out_bf16, void* stream);
/* q,k,v,o bf16 [B, T, heads, head_dim]; head_dim in {72,128} */
DTK_API int dtk_dbg_flash_attn(const void* q, const void* k, const void* v, void* o, int B,
                               int heads, int Tq, int Tk, int head_dim, int causal, int q_pos0,
                               float scale, void* stream);
/* dtk_dbg_flash_attn with grouped KV heads and a borrowed prefix: q, o bf16 [B, Tq, heads, head_dim]; k, v, k2, v2 bf16
 * [B, Tk, kv_heads, head_dim] (query head h reads KV head h / (heads / kv_heads)); key rows below split_row are read from
 * k2 / v2, the others from k / v (split_row = 0: k2 / v2 unused, may be NULL). Returns DTK_ERR_INVALID on bad arguments. */
DTK_API int dtk_dbg_flash_attn_ex(const void* q, const void* k, const void* v, const void* k2, const void* v2, void* o,
                                  int B, int heads, int kv_heads, int Tq, int Tk, int head_dim, int causal, int q_pos0,
                                  int split_row, float scale, void* stream);
/* split-KV single-query decode attention over one layer of a caller-owned slot cache kv bf16
 * [nslots][K | V][kv_heads][max_len][128]. q fp32 [B, heads*128]; slots, pos, share_slot, share_len device int32 [B]
 * (row b attends keys [0, pos[b]]; keys below share_len[b] come from slot share_slot[b]; share_len may be NULL);
 * part_o fp32 [B, heads, 16, 128], part_ml fp32 [B, heads, 16, 2] scratch; counters uint32 [B*heads], zero on entry and
 * zero again on return; out fp32 [B, heads*128], out_bf16 (may be NULL) the same in bf16. nsplit key ranges per (row, head).
 * prefix_len > 0 runs the shared-prefix pass of batched decode first: keys [0, prefix_len) of slot prefix_slot are reduced
 * for all rows by the tensor-core kernel (q_bf16 bf16 [B, heads*128], part_tiles 64-key tiles per CTA) into partial slots
 * [nsplit, nsplit + csplit), csplit = ceil(ceil(prefix_len / 64) / part_tiles), and the per-row pass covers
 * [prefix_len, pos[b]]. B <= 64, nsplit + csplit <= 16, pos[b] >= prefix_len; row state is checked on the host (the call
 * synchronises `stream`). Returns DTK_ERR_INVALID on bad arguments. */
DTK_API int dtk_dbg_decode_attn(const float* q, const void* kv, int nslots, const int* slots, const int* pos,
                                const int* share_slot, const int* share_len, int B, int heads, int kv_heads, int max_len,
                                int nsplit, float scale, float* part_o, float* part_ml, unsigned int* counters,
                                float* out, void* out_bf16, const void* q_bf16, int prefix_slot, int prefix_len,
                                int part_tiles, void* stream);
/* ViT attention on tcgen05: qkv bf16 [B*N, 3*heads*72] (q | k | v column blocks), vt_scratch bf16 [B*heads*80, ceil(N/128)*128],
 * o bf16 [B*N, heads*72]; non-causal, head_dim 72 */
DTK_API int dtk_dbg_attn_tc(const void* qkv, void* vt_scratch, void* o, int B, int heads, int N, float scale, void* stream);
/* y = W[N,K] * rmsnorm?(x[K]) ; mode 0 store / 1 add / 2 glu (out[N/2]) */
DTK_API int dtk_dbg_gemv(const void* W_bf16, const float* x, const void* norm_w_bf16, float eps,
                         int N, int K, int mode, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DETIKZIFY_B200_H */
