/* sutro_b200 — C-ABI of the B200-native local backend for sutro.infer().
 *
 * The reference SDK (sutro-sh/sutro) has no FFI: Sutro.infer() serialises the
 * column and POSTs it to a hosted service (sutro/sdk.py:195-223).  This header
 * is therefore the boundary a maintainer would bind *instead of* that POST; each
 * entry point names the reference interface it stands in for.  INTEGRATION.md
 * shows the ctypes stub that replaces `do_request("POST", "batch-inference")`.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from sb200_last_error() (thread-local, never NULL);
 *   - nothing throws across the boundary;
 *   - "device pointer" arguments are raw CUDA device addresses (PyTorch tensors'
 *     data_ptr() on the Python side); `stream` is a cudaStream_t passed as void*;
 *   - strings travel Arrow-style: one byte blob + int64 offsets[n+1];
 *   - the caller owns inputs; kernel- and engine-level calls write into caller-allocated
 *     device buffers; sb200_infer_text() returns host buffers the library owns until
 *     sb200_result_free().
 */
#ifndef SUTRO_B200_H_
#define SUTRO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB200_ABI_VERSION 1

const char* sb200_last_error(void);
int sb200_abi_version(void);
int sb200_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem);

/* ------------------------------------------------------------------------
 * Kernel-level entry points (used by the parity tests; the engine calls the
 * same launchers internally).  Shapes are in elements, tensors are row-major.
 * ---------------------------------------------------------------------- */

/* epilogue selectors for sb200_gemm_bf16_tn */
#define SB200_EPI_STORE_BF16 0    /* D = bf16(A W^T)                              */
#define SB200_EPI_RESIDUAL_BF16 1 /* D = bf16(bf16(A W^T) + R)                    */
#define SB200_EPI_SWIGLU_BF16 2   /* D[:,j] = silu(acc[:,2j]) * acc[:,2j+1]       */
#define SB200_EPI_STORE_F32 3     /* D = A W^T in fp32 (logits)                   */

/* K1: D[M,N] = A[M,K] W[N,K]^T on tcgen05 tensor cores.  A may be the head of a
 * larger buffer with a_rows >= M rows.  block_n: 0 = auto, else 64/128/256. */
int sb200_gemm_bf16_tn(const void* a, int a_rows, const void* w, void* d, const void* resid, int M,
                       int N, int K, int ldd, int epilogue, int block_n, void* stream);

/* K1+K5 fused: qkv = A Wqkv^T with per-head q/k RMSNorm + RoPE + paged K/V write applied in
 * the GEMM epilogue (same result as sb200_gemm_bf16_tn followed by sb200_rope_kv_write);
 * q heads land in qkv_out[:, :hq*128], K/V go straight to the cache.  block_n: 0/128/256/512. */
int sb200_gemm_qkv_rope(const void* a, int a_rows, const void* w, void* qkv_out, int M, int K,
                        int block_n, const void* q_norm_w, const void* k_norm_w,
                        const void* cos_tab, const void* sin_tab, const int32_t* tok_slot,
                        const int32_t* tok_pos, const int32_t* page_table, int max_pages,
                        void* kv_layer, int hq, int hkv, float eps, void* stream);

/* K4: out = w * bf16(x * rsqrt(mean(x^2)+eps))  (transformers Qwen3RMSNorm) */
int sb200_rmsnorm(const void* x, const void* w, void* out, int rows, int d, float eps,
                  void* stream);

/* K9: embedding gather and the embedding-model head (L2-normalised fp32 rows) */
int sb200_embed_gather(const int32_t* ids, const void* table, void* out, int rows, int d,
                       void* stream);
int sb200_l2_normalize_rows(const void* x, float* out, int rows, int d, void* stream);

/* K5: per-head q/k RMSNorm (NULL weights = none) + RoPE, K/V scatter into the
 * paged cache pool[page][kv_head][K|V][16][128] (swizzled, see DESIGN.md). */
int sb200_rope_kv_write(void* qkv, const void* q_norm_w, const void* k_norm_w, const void* cos_tab,
                        const void* sin_tab, const int32_t* tok_slot, const int32_t* tok_pos,
                        const int32_t* page_table, int max_pages, void* kv_layer, int T, int hq,
                        int hkv, float eps, void* stream);

/* Attention entry points (K2, K3): head_dim 128; hq must be a multiple of hkv with a GQA
 * group hq/hkv of 1, 2, 4, 5 or 8.  Any other group returns -1 and sb200_last_error() names
 * it ("unsupported GQA group size"). */

/* K2: paged-KV decode attention, one query token per sequence. */
int sb200_attn_decode(const void* qkv, void* out, const void* kv_layer, const int32_t* page_table,
                      int max_pages, const int32_t* row_slot, const int32_t* ctx_len, int B, int hq,
                      int hkv, float scale, void* stream);

/* test hook: 0 = automatic choice, 1 = 4-warps-per-pair split kernel, 2 = warp-per-pair */
void sb200_attn_decode_force_variant(int v);

/* K3: causal varlen prefill attention over the paged cache. */
int sb200_attn_prefill(const void* qkv, void* out, const void* kv_layer, const int32_t* page_table,
                       int max_pages, const int32_t* work, int n_work, const int32_t* seq_slot,
                       const int32_t* seq_q_start, const int32_t* seq_q_len,
                       const int32_t* seq_past, int hq, int hkv, float scale, void* stream);
/* tokens per prefill work item (q tile): 128 / (hq/hkv), e.g. 25 for group 5 */
int sb200_attn_prefill_q_tile(int hq, int hkv);

/* K3 on tcgen05 tensor cores (the engine's prefill path): causal varlen attention over DENSE
 * K/V.  qkv:[t_rows, (hq+2*hkv)*128] holds q AND the post-norm/RoPE k, v of the new tokens
 * (what sb200_gemm_qkv_rope leaves there); prefix_kv:[n_layers, prefix_rows, 2*hkv*128]
 * (K heads | V heads) holds the shared prefix, NULL when no sequence has a past.
 * items:[n_items] {seq, q_tile_start}; sequence i attends to prefix rows [0, seq_past[i])
 * and to its own rows [seq_q_start[i], +seq_q_len[i]) causally. */
int sb200_attn_prefill_dense(const void* qkv, int t_rows, void* out, const void* prefix_kv,
                             int prefix_rows, int n_layers, int layer, const int32_t* items,
                             int n_items, const int32_t* seq_q_start, const int32_t* seq_q_len,
                             const int32_t* seq_past, int hq, int hkv, float scale, void* stream);

/* K8: token-level mask of a byte DFA compiled from output_schema. */
int sb200_fsm_build_mask(const int32_t* fsm_trans, const uint8_t* fsm_accept, int n_states,
                         const uint8_t* tok_bytes, const int32_t* tok_off, int vocab, int eos_id,
                         uint32_t* mask_bits, int mask_words, void* stream);

/* K7: batched byte-level BPE on the GPU.  merges:[n,2] left/right ids in rank order
 * (merged_ids NULL => id 256+rank); cls_table: 0x110000 bytes, Unicode class per code
 * point (0 other, 1 letter, 2 number, 3 white space); digits: max digits per pre-token
 * (1 Qwen, 3 Llama-3); tok_bytes/tok_off: vocabulary byte strings (host pointers).
 * encode/decode take DEVICE pointers; out_tokens_dev needs capacity n_bytes;
 * decode with out_bytes_dev == NULL only fills row_byte_off_dev (sizing pass). */
int sb200_tokenizer_create(const int32_t* merges, int n_merges, const int32_t* merged_ids,
                           const uint8_t* cls_table, int digits, const uint8_t* tok_bytes,
                           const int32_t* tok_off, int vocab, void** out);
/* `ignore_merges` of a tokenizer file (tokenizers' BPE: a pre-token that is itself in the
 * vocabulary is emitted as that token without running the merges; Llama-3 files set it).
 * The caller lists the vocabulary entries whose merges do NOT rebuild them: entry ids[i] and the
 * token sequence seq_tokens[seq_off[i] .. seq_off[i+1]) its merges produce (2..32 tokens).  A
 * pre-token that merges to one of these sequences is then emitted as ids[i].  n = 0 clears.
 * Host pointers. */
int sb200_tokenizer_set_word_overrides(void* tok, const int32_t* seq_tokens, const int32_t* seq_off,
                                       const int32_t* ids, int n);
void sb200_tokenizer_destroy(void* tok);
int sb200_tokenizer_encode(void* tok, const uint8_t* text_dev, int64_t n_bytes,
                           const int64_t* row_off_dev, int64_t n_rows, int32_t* out_tokens_dev,
                           int64_t* row_tok_off_dev, void* stream);
int sb200_tokenizer_decode(void* tok, const int32_t* toks_dev, int64_t n_tok,
                           const int64_t* row_tok_off_dev, int64_t n_rows, uint8_t* out_bytes_dev,
                           int64_t* row_byte_off_dev, void* stream);

/* ------------------------------------------------------------------------
 * Engine-level entry points: the local replacement for the hosted service
 * behind `POST batch-inference` / `POST job-results` (sutro/sdk.py:223, :384).
 * One engine per GPU, driven from one host thread.
 * ---------------------------------------------------------------------- */
typedef struct {
  /* architecture */
  int n_layers, d_model, n_q_heads, n_kv_heads, d_ff, vocab, max_position;
  float rms_eps;
  int qk_norm;          /* Qwen3 per-head q/k RMSNorm                                  */
  int embedding_model;  /* prefill-only: last-token pool + L2 normalise                */
  int eos_id;
  /* capacity */
  int max_slots;          /* rows decoded concurrently                                 */
  int max_prefill_tokens; /* new tokens per prefill forward                            */
  int logit_chunk_rows;   /* lm_head / sampling rows per pass (bounds the fp32 logits) */
  int min_admit_rows;     /* free slots to accumulate before interleaving a prefill    */
  int64_t num_pages;      /* KV pool size in 16-token pages (all layers, all kv heads) */
} sb200_engine_config;

typedef struct {          /* device pointers, bf16, layouts as in sutro_b200/modelspec.py */
  const void* embed;      /* [vocab, d_model]                                          */
  const void* lm_head;    /* [vocab, d_model] (== embed when tied)                     */
  const void* final_norm; /* [d_model]                                                 */
  const void* rope_cos;   /* [max_position, 64]                                        */
  const void* rope_sin;
  const void* const* ln1; /* per layer [d_model]                                       */
  const void* const* ln2;
  const void* const* wqkv; /* per layer [(hq+2hkv)*128, d_model], rows q|k|v            */
  const void* const* wo;   /* per layer [d_model, hq*128]                               */
  const void* const* wgu;  /* per layer [2*d_ff, d_model], rows interleaved gate,up     */
  const void* const* wd;   /* per layer [d_model, d_ff]                                 */
  const void* const* q_norm; /* per layer [128] (qk_norm only)                          */
  const void* const* k_norm;
} sb200_engine_weights;

/* progress record — same fields the reference streams from `stream-job-progress`
 * (sutro/sdk.py:331-358): rows done, input tokens, output tokens. */
typedef void (*sb200_progress_fn)(int64_t rows_done, int64_t input_tokens, int64_t output_tokens,
                                  void* user);

typedef struct {
  /* inputs: one prompt per row = prefix_tokens | row tokens | suffix_tokens
   * (stands in for payload["inputs"] + payload["system_prompt"], sutro/sdk.py:196-208) */
  const int32_t* row_tokens_dev;  /* device: all rows' token ids, concatenated          */
  const int64_t* row_tok_off_dev; /* device: [n_rows+1]                                 */
  const int64_t* row_tok_off;     /* host copy of the same offsets                      */
  int64_t n_rows;
  const int32_t* prefix_tokens;   /* host */
  int n_prefix;
  const int32_t* suffix_tokens;   /* host */
  int n_suffix;
  int share_prefix;               /* reuse the prefix KV across rows (page granular)    */
  int max_new_tokens;
  int ignore_eos;
  int truncate_rows;              /* payload["truncate_rows"], sutro/sdk.py:205          */
  /* output_schema automaton (payload["json_schema"]), host arrays; fsm_states 0 = none */
  const int32_t* fsm_trans;       /* [fsm_states, 256], -1 = dead                       */
  const uint8_t* fsm_accept;
  const uint8_t* fsm_final;
  int fsm_states;
  int fsm_start;                  /* state after the forced prefix when n_forced_prefix > 0  */
  /* jump-forward decoding (optional): the last n_forced_prefix tokens of suffix_tokens are
   * output the automaton forces on every row (fed with the prompt, reported as output);
   * fsm_tail_off[fsm_states+1] / fsm_tail_tok give, per state, the tokens of a continuation
   * that is forced all the way to a final state (appended without running the model). */
  int n_forced_prefix;
  const int32_t* fsm_tail_off;    /* host, NULL = no tails */
  const int32_t* fsm_tail_tok;    /* host */
  /* outputs, device, caller-allocated (results["outputs"], sutro/sdk.py:406)           */
  int32_t* out_tokens_dev;        /* [n_rows, max_new_tokens]                           */
  int32_t* out_len_dev;           /* [n_rows]                                           */
  float* out_embed_dev;           /* [n_rows, d_model] (embedding models)               */
  sb200_progress_fn progress;     /* may be NULL                                        */
  void* progress_user;
  int profile;                    /* 1: time every kernel launch with CUDA events        */
  float* out_first_logits_dev;    /* optional [n_rows, vocab]: fp32 logits of each row's first
                                     decision (teacher-forced parity checks); NULL = off   */
  /* payload["sampling_params"] / payload["random_seed_per_input"] (sutro/sdk.py:203-204)  */
  float temperature;              /* 0 = greedy                                          */
  int top_k;                      /* <= 0 = off                                          */
  float top_p;                    /* >= 1 = off (0 is treated as off too)                */
  uint64_t seed;
  int seed_per_row;               /* 1: every row draws from its own Philox stream       */
  float* out_cum_logprob_dev;     /* optional [n_rows]: sum of log p(token) under the masked
                                     softmax at the sampling temperature; NULL = off      */
  const int64_t* row_ids_dev;     /* optional device [n_rows]: the id that keys a row's Philox
                                     stream when seed_per_row = 1 (the row's index in the whole
                                     job when the job is sharded over GPUs, so that draws do not
                                     depend on the sharding); NULL = the local row index       */
} sb200_job;

/* kernel classes for the per-class launch counts / device times in sb200_job_stats */
enum {
  SB200_KC_GEMM = 0,
  SB200_KC_ATTN_DECODE = 1,
  SB200_KC_ATTN_PREFILL = 2,
  SB200_KC_NORM = 3,
  SB200_KC_ROPE = 4,
  SB200_KC_SAMPLE = 5,
  SB200_KC_EMBED = 6,
  SB200_KC_OTHER = 7,
  SB200_KC_COUNT = 8
};

typedef struct {
  int64_t rows_done, input_tokens, prefill_tokens, decode_tokens;
  int64_t prefill_steps, decode_steps, rows_truncated, prefix_cached_tokens;
  int64_t kernel_launches[SB200_KC_COUNT]; /* always filled                              */
  double kernel_ms[SB200_KC_COUNT];        /* device time per class (job.profile only)    */
  double gemm_flops;                       /* 2*M*N*K summed over every GEMM launch       */
  double attn_decode_bytes;                /* K/V bytes the decode attention had to read  */
  /* sb200_infer_text only: CUDA-event times on the engine's stream.  h2d = the rows' bytes and
   * offsets host -> HBM; device = tokenise -> prefill/decode -> detokenise with inputs and
   * outputs resident in HBM; d2h = result buffers HBM -> host.                                */
  double t_h2d_ms, t_device_ms, t_d2h_ms;
} sb200_job_stats;

int sb200_engine_create(const sb200_engine_config* cfg, const sb200_engine_weights* w, void** out);
void sb200_engine_destroy(void* engine);
/* vocabulary byte strings (host): needed for output_schema masks and state advance */
int sb200_engine_set_vocab(void* engine, const uint8_t* tok_bytes, const int32_t* tok_off);
/* blocking; returns when every row has finished (non-zero: see sb200_last_error) */
int sb200_engine_run(void* engine, const sb200_job* job, sb200_job_stats* stats);
void* sb200_engine_stream(void* engine);
/* what a host needs to size buffers: the engine's CUDA device ordinal, whether it is an
 * embedding model (prefill only), d_model and the vocabulary size (any pointer may be NULL) */
int sb200_engine_info(void* engine, int* device, int* embedding_model, int* d_model, int* vocab);

/* ------------------------------------------------------------------------
 * The whole path in one call, HOST buffers in and out — what a non-Python host binds in
 * place of `POST batch-inference` + `POST job-results` (sutro/sdk.py:223, :384-406).
 * rows_bytes / rows_offsets[n_rows+1] are payload["inputs"] Arrow-style (sutro/sdk.py:197);
 * `options` is an sb200_job whose prompt framing (prefix/suffix tokens), schema automaton,
 * max_new_tokens, truncate_rows and sampling fields are used as given — its row-token,
 * output and progress-independent device fields are ignored and filled in here.  The call
 * copies the rows to HBM, tokenises, runs the engine, compacts and detokenises the outputs
 * and copies them back; `*out` is owned by the library until sb200_result_free().
 * results["outputs"][i] (sutro/sdk.py:406) = bytes[offsets[i] .. offsets[i+1]).
 * ---------------------------------------------------------------------- */
typedef struct {
  int64_t n_rows;
  uint8_t* bytes;          /* UTF-8 of all outputs, concatenated (NULL when want_text = 0)   */
  int64_t* offsets;        /* [n_rows+1] into bytes                                          */
  int32_t* tokens;         /* generated token ids, concatenated                               */
  int64_t* token_offsets;  /* [n_rows+1] into tokens                                          */
  float* cum_logprob;      /* [n_rows] (results["cumulative_logprobs"]) or NULL               */
  float* embeddings;       /* [n_rows, d_model] for embedding models, else NULL               */
  int d_model;
} sb200_result;

int sb200_infer_text(void* engine, void* tokenizer, const uint8_t* rows_bytes,
                     const int64_t* rows_offsets, int64_t n_rows, const sb200_job* options,
                     int want_text, int want_logprobs, sb200_result** out,
                     sb200_job_stats* stats);
void sb200_result_free(sb200_result* result);

/* ------------------------------------------------------------------------
 * output_schema -> automaton, natively.  The reference sends the JSON schema itself to its
 * service (payload["json_schema"], sutro/sdk.py:199; built by normalize_output_schema,
 * sutro/common.py:152-163).  sb200_schema_compile takes that JSON text and returns the byte
 * DFA the engine consumes (sb200_job.fsm_trans / fsm_accept / fsm_final); caps for unbounded
 * strings / arrays / integers come from sb200_fsm_limits (NULL = defaults).  Supported:
 * objects with declared properties or free keys (additionalProperties maps), strings
 * (min/maxLength; formats date, time, date-time, uuid, email, uri, ipv4, duration), integer / number bounds and multipleOf,
 * booleans, null,
 * arrays (items, min/maxItems, prefixItems tuples, uniqueItems over small enumerations), enum,
 * const, anyOf / oneOf, compatible allOf, $ref into $defs, type lists.  A keyword outside that
 * set (pattern, ...) that would constrain the
 * output is an error (-2 = argument error), never ignored.  The tables stay owned by the
 * schema handle until sb200_schema_destroy.
 * ---------------------------------------------------------------------- */
typedef struct {
  int max_string_chars; /* cap when a string has no maxLength (default 64)      */
  int max_array_items;  /* cap when an array has no maxItems (8)                 */
  int max_int_digits;   /* digits of an unbounded integer (9)                    */
  int max_frac_digits;  /* fraction digits of a number (4)                       */
  int small_int_range;  /* integer ranges up to this size are enumerated (2048)  */
  int max_recursion;    /* how often a recursive $ref may be re-entered (2)      */
} sb200_fsm_limits;

void sb200_fsm_limits_default(sb200_fsm_limits* limits);
int sb200_schema_compile(const char* json_utf8, int64_t len, const sb200_fsm_limits* limits,
                         void** out_schema);
void sb200_schema_destroy(void* schema);
int sb200_schema_tables(void* schema, const int32_t** trans, const uint8_t** accept,
                        const uint8_t** final_states, int* n_states, int* start);
/* bytes of the longest accepted string (an upper bound on the tokens a constrained row can
 * need), -1 when the language is unbounded */
int64_t sb200_schema_longest_path(void* schema);

/* ------------------------------------------------------------------------
 * A model on disk and the strings-only call: the whole request of the reference's
 * `POST batch-inference` payload — model, inputs, system_prompt, json_schema, sampling_params
 * (sutro/sdk.py:196-208) — served without any Python on the host side.
 *
 * sb200_model_open reads a bundle directory written by `python -m sutro_b200.bundle`
 * (manifest.json + data.bin: architecture, bf16 weights in the engine's layout, RoPE tables,
 * tokenizer tables, special-token ids, template family), uploads the weights and creates the
 * engine and the GPU tokenizer.  max_slots / max_prefill_tokens / kv_pages <= 0 pick defaults
 * (512 / 8192 / 80 % of the free memory).
 *
 * sb200_model_infer renders the chat template around `system_prompt_utf8` (NULL/"" = none),
 * compiles `json_schema_utf8` (NULL = unconstrained) with sb200_schema_compile, derives the
 * jump-forward plan from the automaton, picks max_new_tokens when <= 0 (the longest string the
 * schema admits, else 512; capped at half the context window) and runs sb200_infer_text on the
 * rows.  `sampling` may be NULL (greedy); only its temperature / top_k / top_p / seed /
 * seed_per_row / ignore_eos / truncate_rows / progress fields are read.
 * ---------------------------------------------------------------------- */
int sb200_model_open(const char* bundle_dir, int device, int max_slots, int max_prefill_tokens,
                     int64_t kv_pages, void** out_model);
void sb200_model_close(void* model);
void* sb200_model_engine(void* model);
void* sb200_model_tokenizer(void* model);
int sb200_model_infer(void* model, const char* system_prompt_utf8, const char* json_schema_utf8,
                      int64_t schema_len, const sb200_fsm_limits* limits, int max_new_tokens,
                      const sb200_job* sampling, const uint8_t* rows_bytes,
                      const int64_t* rows_offsets, int64_t n_rows, int want_logprobs,
                      sb200_result** out, sb200_job_stats* stats);

/* Device-side Arrow helpers used by the Python host instead of tensor-library ops.
 * compact_rows: out_tokens[n_rows, stride] with len[i] valid tokens per row -> off[n_rows+1]
 * and the flat token array (capacity n_rows*stride).
 * rows_select: pick m rows of a device-resident string column by index (row sharding across
 * GPUs; the ordered gather of per-rank results on rank 0: results["outputs"] stay positional,
 * sutro/sdk.py:406-412).  The source may be a batch of equally strided columns — row j is row
 * j % part_rows of part j / part_rows, whose offsets start at off[part*(part_rows+1)] and whose
 * bytes start at bytes + part*part_bytes (what a gather of padded per-rank buffers looks like);
 * a plain column is part_rows = its row count, part_bytes = 0.  out_bytes needs room for the
 * selected rows (the source size always suffices). */
int sb200_compact_rows(const int32_t* out_tokens_dev, const int32_t* out_len_dev, int64_t n_rows,
                       int stride, int64_t* off_dev, int32_t* flat_dev, void* stream);
int sb200_rows_select(const uint8_t* bytes_dev, const int64_t* off_dev, int64_t part_rows,
                      int64_t part_bytes, const int64_t* idx_dev, int64_t m, int64_t* out_off_dev,
                      uint8_t* out_bytes_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SUTRO_B200_H_ */
