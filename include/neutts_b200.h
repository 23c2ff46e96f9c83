/* neutts_b200 — C-ABI of the B200 (sm_100a) implementation of NeuTTS-Air's two inference
 * hot paths.  Plain pointers and sizes only; no torch / C++ types cross this boundary.
 *
 * The reference has no FFI of its own (it is 465 lines of Python over `transformers` and
 * `neucodec`); the two inner seams this library replaces are
 *
 *   seam 1 (speech LM)  neutts/neutts.py:334-352  NeuTTS._infer_torch ->
 *                       self.backbone.generate(prompt, max_length=2048, eos_token_id=...,
 *                       do_sample=True, temperature=1.0, top_k=50, use_cache=True,
 *                       min_new_tokens=50)                     -> nt_lm_prefill + nt_lm_decode
 *   seam 2 (codec)      neutts/neutts.py:273-295  NeuTTS._decode ->
 *                       self.codec.decode_code(codes[B,1,N]) -> float[B,1,480N]
 *                                                              -> nt_codec_decode
 *
 * Conventions
 *   - every function returns 0 on success, a negative nt_status otherwise; nt_last_error()
 *     returns a human-readable message for the calling thread's last failure;
 *   - all device memory (weights, KV pages, workspaces, inputs, outputs) is allocated and
 *     owned by the caller (the Python shim uses torch tensors); the library never frees it;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream
 *     unless stated otherwise;
 *   - matrices are row-major [out_features, in_features] exactly as torch.nn.Linear stores
 *     them; "bf16" means __nv_bfloat16, "f32" float.
 */
#ifndef NEUTTS_B200_H_
#define NEUTTS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  NT_OK = 0,
  NT_ERR_INVALID = -1,   /* bad argument / unsupported shape  -> ValueError in the shim  */
  NT_ERR_CUDA = -2,      /* CUDA runtime / driver failure     -> RuntimeError            */
  NT_ERR_NOMEM = -3,     /* caller-provided workspace too small                          */
  NT_ERR_STATE = -4      /* call order violated (e.g. decode before prefill)             */
} nt_status;

const char* nt_last_error(void);
/* library/ABI version, bumped on any signature change */
int nt_abi_version(void);   /* 2: nt_sampling gained limits + slot_base; 3: nt_codec_config.precision */
/* number of kernels launched by this library since load (all streams); bench.py reports the delta */
uint64_t nt_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Generic tensor-core GEMM (tcgen05 + TMEM + TMA):  C[M,N] = epilogue(A[M,K] . W[N,K]^T)
 * Used by prefill, batched decode and the codec.  Replaces torch addmm/mm as reached from
 * transformers modeling_qwen2.py:46-48,217-219,244,475 and the codec's Linear/Conv1d layers.
 * ------------------------------------------------------------------------------------------ */
typedef enum { NT_BF16 = 0, NT_TF32 = 1 } nt_dtype;          /* A/W element type: bf16, or f32 fed as tf32 */
typedef enum { NT_ACT_NONE = 0, NT_ACT_SILU = 1, NT_ACT_SWIGLU = 2 } nt_act;

typedef struct {
  nt_dtype dtype;
  int M, N, K;
  const void* A;      /* [M, K] elements, row stride lda (elements).  lda < K is allowed: rows
                         then overlap, which is how Conv1d is expressed (im2col as a view)   */
  int64_t lda;
  const void* W;      /* [N, K], row stride ldw */
  int64_t ldw;
  const float* bias;      /* [N] or NULL */
  const float* residual;  /* [M, ldr] f32 or NULL; may alias out_f32 */
  int64_t ldr;
  nt_act act;             /* SWIGLU: columns (2j, 2j+1) = (gate_j, up_j) -> one output column j */
  float* out_f32;         /* [M, ldc] or NULL */
  void* out_bf16;         /* [M, ldc] or NULL */
  int64_t ldc;
  /* row mask for padded-batch layouts: if valid_period > 0 only rows with
     (row % valid_period) < valid_len are written */
  int valid_period, valid_len;
} nt_gemm_args;

int nt_gemm(const nt_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * Speech LM (seam 1)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int vocab_size, hidden, inter, n_layers, n_heads, n_kv_heads, head_dim; /* head_dim must be 64 */
  float rms_eps, rope_theta;
  int max_batch;      /* sequences resident at once */
  int max_ctx;        /* context limit (prompt + generated), reference: 2048 (neutts.py:85) */
  int page_size;      /* KV page, tokens; must be 64 */
  int num_pages;      /* pages in the pool (shared by all layers: one page id addresses every layer) */
  int max_prefill_tokens; /* sum of prompt lengths per nt_lm_prefill call */
} nt_lm_config;

/* Device pointers.  Packed layouts (built by neutts_air_b200/lm.py:pack_weights):
 *   wqkv  [ (n_heads+2*n_kv_heads)*64, hidden ] bf16, rows ordered q heads, k heads, v heads;
 *         inside every q/k head the 64 rows are interleaved (0,32,1,33,...,31,63) so RoPE
 *         partners are adjacent; v heads keep natural order.  bqkv follows the same order.
 *   wgu   [ 2*inter, hidden ] bf16, rows interleaved (gate_0, up_0, gate_1, up_1, ...).
 *   wo    [ hidden, n_heads*64 ],  wd [ hidden, inter ],  embed / lm_head [ vocab, hidden ].
 * The per-layer arrays are host arrays of n_layers device pointers. */
typedef struct {
  const void* embed;
  const void* lm_head;
  const float* final_norm;
  const float* const* ln1;
  const void* const* wqkv;
  const float* const* bqkv;
  const void* const* wo;
  const float* const* ln2;
  const void* const* wgu;
  const void* const* wd;
} nt_lm_weights;

/* Caller-owned device state for a batch of sequences (slots 0..B-1). */
typedef struct {
  void* kv_pages;        /* bf16 [n_layers][2 (k,v)][num_pages][n_kv_heads][page_size][64] */
  int32_t* page_table;   /* [max_batch][max_ctx/page_size] page ids */
  int32_t* seq_lens;     /* [max_batch] tokens already in the KV cache */
  int32_t* cur_token;    /* [max_batch] last sampled token (input of the next decode step) */
  int32_t* out_tokens;   /* [max_batch][max_new] generated ids (includes the EOS if hit) */
  int32_t* n_generated;  /* [max_batch] */
  int32_t* done;         /* [max_batch] 1 once EOS sampled or max_ctx reached */
  int32_t max_new;       /* row length of out_tokens */
} nt_lm_state;

/* Sampling semantics of transformers generation (logits_process.py:224-233,296-299,580-586;
 * utils.py:2789-2791): EOS masked while n_generated < min_new_tokens, logits / temperature,
 * keep the top_k largest, softmax, one multinomial draw (Philox4x32-10 keyed by seed, slot, step). */
typedef struct {
  int32_t eos_id;
  int32_t min_new_tokens;
  int32_t max_new_tokens;   /* stop after this many generated tokens (<= state.max_new) */
  int32_t top_k;            /* 1..64 */
  float temperature;
  uint64_t seed;
  int32_t greedy;           /* 1: argmax instead of sampling (tests) */
  const int32_t* forced;    /* optional [max_batch][max_new] teacher-forced tokens (tests), else NULL */
  const int32_t* limits;    /* optional device [max_batch]: per-sequence cap on generated tokens (transformers'
                               max_length is prompt + generated PER SEQUENCE, stopping_criteria.py:73-84), else NULL */
  int32_t slot_base;        /* global index of slot 0: keys the Philox stream, so chunks / ranks draw independently */
} nt_sampling;

typedef struct nt_lm nt_lm;

size_t nt_lm_workspace_bytes(const nt_lm_config* cfg);
int nt_lm_create(const nt_lm_config* cfg, const nt_lm_weights* w, void* workspace, size_t workspace_bytes, nt_lm** out);
int nt_lm_destroy(nt_lm* lm);

/* Prefill B prompts packed back to back: ids [total] (device), cu_seqlens [B+1] (host).
 * Fills the KV cache, samples the first token of every sequence (A2 + A10-A12 of SURVEY §8a).
 * logits_out: optional device f32 [B][vocab] receiving the last-position logits. */
int nt_lm_prefill(nt_lm* lm, const nt_lm_state* st, const int32_t* ids, const int32_t* cu_seqlens_host, int B,
                  const nt_sampling* sp, float* logits_out, void* stream);

/* Run n_steps decode steps for slots 0..B-1 with no host synchronisation in between
 * (finished slots keep their state; their work is skipped on device).
 * logits_out: optional device f32 [n_steps][B][vocab] (tests only; forces logits to HBM). */
int nt_lm_decode(nt_lm* lm, const nt_lm_state* st, int B, int n_steps, const nt_sampling* sp, float* logits_out,
                 void* stream);

/* Timed single-kernel entry for the roofline measurement: the lm_head GEMV (+ final RMSNorm)
 * exactly as the decode step launches it.  h: f32 [B][hidden] -> logits f32 [B][vocab]. */
int nt_lm_head_gemv(nt_lm* lm, const float* h, int B, float* logits, void* stream);

/* Per-stage parity hooks (tests): run only the first n_layers layers (-1 = all), and look up an
 * internal activation buffer by name ("h", "q", "qkv", "attn", "act", "logits", "xn", "attn_bf16",
 * "act_bf16", "h_last"); the pointer lies inside the caller's workspace. */
int nt_lm_debug_set_layers(nt_lm* lm, int n_layers);
/* launch-latency probe: n dependent trivial kernels (grid x block) each incrementing *counter */
int nt_debug_launch_chain(int n, int grid, int block, int* counter, void* stream);
void* nt_lm_debug_ptr(nt_lm* lm, const char* name);
/* megakernel timeline: buf = device int64 [2][1024] receiving %globaltimer marks of decode step `step`
 * from the first and the last CTA (NULL disables) */
int nt_lm_debug_set_profile(nt_lm* lm, long long* buf, int step);

/* ------------------------------------------------------------------------------------------
 * NeuCodec decoder (seam 2)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int hidden, depth, heads, head_dim;   /* 1024, 12, 16, 64 */
  int mlp_hidden;                       /* 4096 */
  int groups;                           /* GroupNorm groups (32) */
  int embed_kernel;                     /* 7 */
  int n_fft, hop;                       /* 1920, 480 */
  int fsq_levels, fsq_dims;             /* 4, 8 */
  float norm_eps, rope_base, mag_clip;
  int rope_time_axis;                   /* 1: rotary over frames; 0: upstream quirk (no-op, skipped) */
  int max_batch, max_frames;
  int precision;                        /* arithmetic of the tensor-core GEMMs (fp32 storage, fp32 accumulate):
                                           0 = TF32, with 3xTF32 (hi/lo operand split, fp32-grade products) for the ISTFT
                                               head and the inverse-DFT GEMMs only ("mixed")
                                           1 = TF32 everywhere (fastest; 3.4e-4 abs RMS on speech-level weights)
                                           2 = 3xTF32 everywhere (fp32-grade; what the Python host passes by default:
                                               the only mode within 1e-3 RMS of the fp32 path on adversarial heads) */
} nt_codec_config;

/* All f32, device.  Conv weights are pre-flattened tap-major: [C_out, k*C_in] with
 * W2[co, tap*C_in + ci] = W[co, ci, tap].  fsq_w/fsq_b are the collapsed
 * fc_post_a(project_out(.)) affine: [hidden, fsq_dims], [hidden]. */
typedef struct {
  const float* fsq_w; const float* fsq_b;
  const float* embed_w; const float* embed_b;
  /* 4 resnet blocks (2 prior, 2 post): arrays of 4 device pointers each */
  const float* const* rn_n1w; const float* const* rn_n1b; const float* const* rn_c1w; const float* const* rn_c1b;
  const float* const* rn_n2w; const float* const* rn_n2b; const float* const* rn_c2w; const float* const* rn_c2b;
  /* depth transformer blocks */
  const float* const* att_norm; const float* const* wqkv; const float* const* wproj;
  const float* const* ffn_norm; const float* const* fc1; const float* const* fc2;
  const float* final_ln_w; const float* final_ln_b;
  const float* head_w;   /* [n_fft+2, hidden] */
  const float* head_b;
  const float* idft_basis; /* [n_fft, Kpad] f32: windowed inverse-rDFT basis, Kpad = roundup(n_fft+2, 32) */
} nt_codec_weights;

typedef struct nt_codec nt_codec;

size_t nt_codec_workspace_bytes(const nt_codec_config* cfg);
int nt_codec_create(const nt_codec_config* cfg, const nt_codec_weights* w, void* workspace, size_t workspace_bytes,
                    nt_codec** out);
int nt_codec_destroy(nt_codec* c);
/* codes: device int32 [B][N] (all items the same length N); pcm: device f32 [B][hop*N].
 * The same forward pass as nt_codec_decode_ragged with every length N. */
int nt_codec_decode(nt_codec* c, const int32_t* codes, int B, int N, float* pcm, void* stream);
/* Items of different lengths in one forward pass.
 * codes: device int32, items packed back to back: item b = codes[cu_frames[b] .. cu_frames[b+1]);
 * cu_frames: HOST int32 [B+1], cu_frames[0] = 0, every length in 1..max_frames, 1 <= B <= max_batch;
 * pcm: device f32 [hop * cu_frames[B]], item b at pcm[hop*cu_frames[b]] (hop*N_b samples).
 * Asynchronous on `stream` (no host synchronisation); item b's samples equal a decode of item b alone. */
int nt_codec_decode_ragged(nt_codec* c, const int32_t* codes, const int32_t* cu_frames, int B, float* pcm, void* stream);

/* ------------------------------------------------------------------------------------------
 * Single-op entry points (unit tests; each mirrors one row of SURVEY.md §8a)
 * ------------------------------------------------------------------------------------------ */
int nt_op_rmsnorm(const float* x, const float* w, float eps, int rows, int cols, float* out_f32, void* out_bf16,
                  void* stream);
int nt_op_topk_sample(const float* logits, int B, int V, const nt_sampling* sp, const int32_t* n_generated,
                      int32_t step, int32_t* out_token, float* out_topk_val, int32_t* out_topk_idx, void* workspace,
                      size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEUTTS_B200_H_ */
