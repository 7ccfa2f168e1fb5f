/*
 * nano_infer_abi.h -- binary-compatible view of the reference host API (bd4sur/Nano infer/infer.h,
 * infer/tensor.h, infer/tokenizer.h) for libnano_infer_b200.so.
 *
 * Reference products (main_cli.c, main_wss.c, main_sort.c, main_wasm.c, ui_llm.c) are compiled against the
 * reference's OWN headers and only LINKED against our library, so what must match is the ABI: struct layouts
 * (callers read ctx->llm->config.*, llm->arch/quant_type/group_size, ctx->tokenizer->vocab[], write
 * ctx->sampler->temperature/top_p and ctx->observation*: SURVEY finding 8) and the exported prototypes
 * (infer.h:253-282).  tests/test_boundary.py checks every size/offset below against tests/golden/abi_layout.json,
 * the layout read from the reference's own headers (oracle/ref_harness.c:orh_abi_layout).
 *
 * Private areas: nobody outside the reference's infer.c touches LLM.state (FwdBuffer) or LLM.params
 * (grep-verified in SURVEY finding 8); the shim keeps its engine handle and host logits buffer there.
 */
#ifndef NANO_INFER_ABI_H
#define NANO_INFER_ABI_H

#include <stdint.h>
#include <stddef.h>
#include <wchar.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- infer.h:45-55 ---- */
enum { NANO_ARCH_NANO = 0, NANO_ARCH_QWEN2 = 2, NANO_ARCH_QWEN3 = 3 };
enum { NANO_RUN_PREFILL = 11, NANO_RUN_DECODE = 12, NANO_STOP_NORMAL = -10, NANO_STOP_IN_PREFILL = -11,
       NANO_STOP_IN_DECODE = -12, NANO_STOP_ERROR = -20 };
/* ---- infer.h:65-76 observation phases ---- */
enum { NANO_PH_EMBEDDING = 1, NANO_PH_ATTN_NORM, NANO_PH_QKV, NANO_PH_QK_ROPE, NANO_PH_MHA, NANO_PH_O, NANO_PH_FFN_NORM,
       NANO_PH_W1W3, NANO_PH_W2, NANO_PH_FINAL_NORM, NANO_PH_CLASSIFY, NANO_PH_SAMPLE };

/* infer.h:78-87 */
typedef struct Nano_Observation {
    int32_t layer, phase;
    uint32_t token_0, token_1, token_2, token_3, token_4, token_5;
} Nano_Observation;

/* tensor.h:84-90, 143-147 */
typedef struct { int8_t *q; float *s; } Q80_Tensor;
typedef union { uint8_t *tensor_q4k; Q80_Tensor tensor_q80; float *tensor_f32; } Typed_Tensor;

/* infer.h:89-99 */
typedef struct {
    uint32_t block_size, vocab_size, n_layer, n_embd, n_head, n_kv_head, n_hidden, is_shared_classifier, head_dim;
} LLM_Config;

/* infer.h:101-131 : 21 pointers; private to the engine */
typedef struct {
    Typed_Tensor *q_tokens; float *token_embedding;
    float *rms_norm_attn, *rms_norm_ffn, *rms_norm_final;
    Typed_Tensor *wq, *wk, *wv, *wo;
    float *bq, *bk, *bv;
    float *q_norm, *k_norm;
    Typed_Tensor *w1, *w2, *w3;
    float *freq_cis_real, *freq_cis_imag;
    Typed_Tensor *token_classifier;
} LLM_Param;

/* infer.h:133-166 : private to the engine.  The shim uses: xbuf = nb200_engine*, logits = host float[vocab]. */
typedef struct {
    float *xbuf; int8_t *qvbuf; float *qsbuf; float *kvcache;
    float *x, *xb, *xba, *xb2, *hb, *hb2;
    Typed_Tensor xq, xbaq, hq;
    float *q, *k, *v, *k_cache, *v_cache, *att, *logits;
    float *q0, *k0, *v0, *o0, *q1, *k1, *v1, *o1;
} FwdBuffer;

/* infer.h:168-180 */
typedef struct {
    LLM_Config config; LLM_Param params; FwdBuffer state;
    uint32_t arch, quant_type, group_size;
    int fd; uint8_t *buffer; size_t file_size;
} LLM;

/* infer.h:182-207 */
typedef struct { uint32_t lora_rank, lora_alpha, n_layer, n_embd, n_head, n_kv_head, n_hidden, lora_config; } LoRA_Config;
typedef struct { float *wq_lora_a, *wq_lora_b, *wk_lora_a, *wk_lora_b, *wv_lora_a, *wv_lora_b, *wo_lora_a, *wo_lora_b; } LoRA_Param;
typedef struct { LoRA_Config config; LoRA_Param params; float *data; } LoRA;

/* infer.h:209-222 */
typedef struct { float prob; int index; } ProbIndex;
typedef struct {
    int vocab_size; ProbIndex *probindex;
    float repetition_penalty, temperature, top_p; uint32_t top_k; uint64_t rng_state;
} Sampler;

/* tokenizer.h:16-37 */
typedef struct { char *str; int id; } TokenIndex;
struct Trie; struct Map;
typedef struct {
    uint32_t vocab_size;
    wchar_t *unicode_charset; wchar_t **token_list;
    struct Trie *vocab_trie; struct Map *unicode_to_id_map; struct Map *token_to_id_map;
    char **vocab; float *vocab_scores; TokenIndex *sorted_vocab; unsigned int max_token_length;
    unsigned char byte_pieces[512];
} Tokenizer;

/* infer.h:224-234 */
typedef struct Nano_Context {
    LLM *llm; LoRA *lora; Tokenizer *tokenizer; Sampler *sampler;
    uint32_t max_seq_len; uint64_t random_seed;
    void (*observation)(Nano_Observation obs, void *env); void *observation_env;
} Nano_Context;

/* infer.h:236-250 */
typedef struct Nano_Session {
    wchar_t *prompt; uint32_t num_prompt_tokens, max_seq_len; uint32_t *output_ids; uint32_t output_count;
    wchar_t *output_text; uint32_t next_token, pos; int32_t is_prefilling; uint64_t t_0, t_1; float tps;
} Nano_Session;

/* ---- exported by libnano_infer_b200.so: the prototypes of infer.h:253-282 ---- */
void load_llm_from_buffer(LLM *llm, Tokenizer *tk, uint8_t *buffer, uint32_t max_seq_len);
void load_llm(LLM *llm, Tokenizer *tk, char *model_path, uint32_t max_seq_len);
Sampler *build_sampler(int vocab_size, float repetition_penalty, float temperature, float top_p, uint32_t top_k, uint64_t rng_seed);
LoRA *load_lora_from_buffer(LLM *llm, uint8_t *buffer);
LoRA *load_lora(LLM *llm, char *lora_path);
Nano_Context *llm_context_init_from_buffer(uint8_t *buffer, uint32_t max_seq_len, float repetition_penalty, float temperature,
                                           float top_p, uint32_t top_k, uint64_t random_seed);
Nano_Context *llm_context_init(char *model_path, char *lora_path, uint32_t max_seq_len, float repetition_penalty,
                               float temperature, float top_p, uint32_t top_k, uint64_t random_seed);
void llm_context_free(Nano_Context *ctx);
uint32_t generate_next_token(Nano_Context *ctx, uint32_t *output_ids, uint32_t pos, int is_prefilling);
Nano_Session *llm_session_init(Nano_Context *ctx, wchar_t *prompt, uint32_t max_seq_len, int32_t is_thinking_enabled);
int32_t llm_session_step(Nano_Context *ctx, Nano_Session *session);
void llm_session_free(Nano_Session *session);
int32_t generate_sync(Nano_Context *ctx, wchar_t *prompt, uint32_t max_seq_len, int32_t (*on_prefilling)(Nano_Session *),
                      int32_t (*on_decoding)(Nano_Session *), int32_t (*on_finished)(Nano_Session *));
void seq2seq(Nano_Context *ctx, wchar_t *input_list, wchar_t *output_list, uint32_t max_seq_len);
void free_lora(LLM *llm, LoRA *lora);
void free_llm(LLM *llm, Tokenizer *tk);
void free_sampler(Sampler *sampler);
/* un-headered in the reference but non-static (infer.c:971); kept for harnesses: returns HOST logits */
float *llm_forward(Nano_Context *ctx, uint32_t token, uint32_t pos, uint32_t max_seq_len, uint32_t is_causal, LLM *llm, LoRA *lora);

/* ---- tensor.h:153-166 (host-pointer semantics; used by infer/tools/export_q4k.c) ---- */
void dequantize(Q80_Tensor *qx, float *x, int n, uint32_t group_size);
void quantize(Q80_Tensor *qx, float *x, int n, uint32_t group_size);
Typed_Tensor *parse_quantized_tensors(void **ptr, int n, int size_each, uint32_t group_size);
uint64_t bytes_num_of_q4k_tensor(uint8_t *Q);
uint8_t *make_q4k_tensor(uint32_t ndim, uint32_t shape[]);
void dequantize_tensor_q4k(uint8_t *Q, float *t_out, uint32_t *ndim, uint32_t *shape);
uint8_t *pack_q4k_tensor(uint8_t *Q);
uint8_t *unpack_q4k_tensor(uint8_t *buffer, uint64_t *p_total_bytes);
uint8_t *quantize_tensor_q4k(float *t, uint32_t ndim, uint32_t shape[]);                     /* tensor.h:160 */
void quantize_tensor_q4k_in_situ(float *t, uint32_t ndim, uint32_t shape[], uint8_t *T);     /* tensor.h:161 */
void matmul_q4k(float *xout, uint8_t *x, uint8_t *w, uint32_t layer);                        /* tensor.h:166 */
/* The three above run on the GPU (nb200_op_q4k_quantize_blocks / nb200_op_q4k_matvec_blocks) and need last
 * dimensions that are multiples of 256 (the reference's partial-block path is broken, tensor.c:307). */

/* ---- imported from the reference's unchanged host objects at link time (utils.c, tokenizer.c, hal_ram_linux.c) ---- */
void *platform_calloc(size_t n, size_t sizeoftype);
void *platform_malloc(size_t nbytes);
float random_f32(uint64_t *state);
struct Map *new_map(uint32_t bucket_num);
uint32_t map_set(struct Map *m, uint32_t key, uint32_t value);
struct Trie *new_trie(uint32_t vocab_size, uint8_t is_end_of_token);
int add_token(struct Trie *trie, uint32_t *token, uint32_t token_len, uint32_t token_id);
uint32_t *string_to_ids(struct Map *unicode_to_id_map, wchar_t *utext);
void build_bpe_tokenizer(Tokenizer *t, uint8_t *tokenizer_buffer, int vocab_size);
void free_bpe_tokenizer(Tokenizer *t);
void free_tokenizer(Tokenizer *tk);
uint32_t *encode_nano(Tokenizer *t, wchar_t *text, uint32_t *n_tokens_ptr);
wchar_t *decode_nano(Tokenizer *t, uint32_t *ids, uint32_t len);
wchar_t *decode_bpe(Tokenizer *t, uint32_t *ids, uint32_t len);
uint32_t *apply_qwen_chat_template(Tokenizer *t, wchar_t *user_prompt_wchar, uint32_t *prompt_length, int32_t enable_thinking);

#ifdef __cplusplus
}
#endif
#endif
