/*
 * host_stub.c -- a stand-in for the host-side objects a program links beside libnano_infer_b200.so (the imported block
 * at the end of include/nano_infer_abi.h): allocation, the sampler's xorshift generator and a tokenizer.  The tests load
 * it with RTLD_GLOBAL before the shim so that the shim can be called without the original project's host sources.
 *
 * The tokenizer is character-level: encode_nano maps each character through the map the shim fills from the model's
 * single-character tokens, decode_nano concatenates token strings.  That covers the digit prompts the tests use.
 * Multi-character tokens and the BPE tokenizer are accepted and ignored: the Qwen-architecture tests pass token ids.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <wchar.h>

#include "nano_infer_abi.h"

struct Map { uint32_t n, cap; uint32_t *key, *val; };
struct Trie { uint32_t vocab_size; };

void *platform_calloc(size_t n, size_t sizeoftype) { return calloc(n, sizeoftype); }
void *platform_malloc(size_t nbytes) { return malloc(nbytes); }

/* xorshift64* as in llama2.c: the sampler's coin; bit-identical to the stream tests/golden/make_golden.py restates */
float random_f32(uint64_t *state) {
    *state ^= *state >> 12;
    *state ^= *state << 25;
    *state ^= *state >> 27;
    const uint32_t u = (uint32_t)((*state * 0x2545F4914F6CDD1Dull) >> 32);
    return (float)(u >> 8) / 16777216.0f;
}

struct Map *new_map(uint32_t bucket_num) {
    struct Map *m = (struct Map *)calloc(1, sizeof(struct Map));
    m->cap = bucket_num ? bucket_num : 1;
    m->key = (uint32_t *)calloc(m->cap, sizeof(uint32_t));
    m->val = (uint32_t *)calloc(m->cap, sizeof(uint32_t));
    return m;
}

static int map_find(const struct Map *m, uint32_t key) {
    for (uint32_t i = 0; i < m->n; i++) if (m->key[i] == key) return (int)i;
    return -1;
}

uint32_t map_set(struct Map *m, uint32_t key, uint32_t value) {
    int i = map_find(m, key);
    if (i < 0) {
        if (m->n == m->cap) {
            m->cap *= 2;
            m->key = (uint32_t *)realloc(m->key, m->cap * sizeof(uint32_t));
            m->val = (uint32_t *)realloc(m->val, m->cap * sizeof(uint32_t));
        }
        i = (int)m->n++;
        m->key[i] = key;
    }
    m->val[i] = value;
    return value;
}

static void free_map(struct Map *m) {
    if (!m) return;
    free(m->key); free(m->val); free(m);
}

struct Trie *new_trie(uint32_t vocab_size, uint8_t is_end_of_token) {
    (void)is_end_of_token;
    struct Trie *t = (struct Trie *)calloc(1, sizeof(struct Trie));
    t->vocab_size = vocab_size;
    return t;
}

int add_token(struct Trie *trie, uint32_t *token, uint32_t token_len, uint32_t token_id) {
    (void)trie; (void)token; (void)token_len; (void)token_id;
    return 0;
}

uint32_t *string_to_ids(struct Map *unicode_to_id_map, wchar_t *utext) {
    const size_t n = wcslen(utext);
    uint32_t *ids = (uint32_t *)calloc(n + 1, sizeof(uint32_t));
    for (size_t i = 0; i < n; i++) {
        const int j = map_find(unicode_to_id_map, (uint32_t)utext[i]);
        ids[i] = j < 0 ? 0 : unicode_to_id_map->val[j];
    }
    return ids;
}

uint32_t *encode_nano(Tokenizer *t, wchar_t *text, uint32_t *n_tokens_ptr) {
    *n_tokens_ptr = (uint32_t)wcslen(text);
    return string_to_ids(t->unicode_to_id_map, text);
}

wchar_t *decode_nano(Tokenizer *t, uint32_t *ids, uint32_t len) {
    size_t n = 0;
    for (uint32_t i = 0; i < len; i++)
        if (ids[i] < t->vocab_size && t->token_list[ids[i]]) n += wcslen(t->token_list[ids[i]]);
    wchar_t *out = (wchar_t *)calloc(n + 1, sizeof(wchar_t));
    for (uint32_t i = 0; i < len; i++)
        if (ids[i] < t->vocab_size && t->token_list[ids[i]]) wcscat(out, t->token_list[ids[i]]);
    return out;
}

void free_tokenizer(Tokenizer *tk) {
    if (tk->token_list)
        for (uint32_t i = 0; i < tk->vocab_size; i++) free(tk->token_list[i]);
    free(tk->token_list); free(tk->unicode_charset); free(tk->vocab_trie);
    free_map(tk->unicode_to_id_map); free_map(tk->token_to_id_map);
}

void build_bpe_tokenizer(Tokenizer *t, uint8_t *tokenizer_buffer, int vocab_size) {
    (void)tokenizer_buffer;
    t->vocab_size = (uint32_t)vocab_size;
}

void free_bpe_tokenizer(Tokenizer *t) { (void)t; }

wchar_t *decode_bpe(Tokenizer *t, uint32_t *ids, uint32_t len) {
    (void)t; (void)ids; (void)len;
    return (wchar_t *)calloc(1, sizeof(wchar_t));
}

uint32_t *apply_qwen_chat_template(Tokenizer *t, wchar_t *user_prompt_wchar, uint32_t *prompt_length, int32_t enable_thinking) {
    (void)t; (void)user_prompt_wchar; (void)enable_thinking;
    *prompt_length = 1;
    return (uint32_t *)calloc(1, sizeof(uint32_t));
}
