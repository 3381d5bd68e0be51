/*
 * vibrato_b200.h — C ABI of the B200-native batched Viterbi tokenizer.
 *
 * The reference (daac-tools/vibrato, Rust) has no FFI; its seam is the public Rust API consumed by
 * the `tokenize` and `benchmark` crates (SURVEY.md §8b).  Each entry point below names the Rust
 * item it stands behind (paths relative to /root/reference/vibrato/src/); INTEGRATION.md shows the
 * Rust shim (`extern "C"` block + Dictionary/Tokenizer/Worker/Token wrappers) that binds them.
 *
 * Conventions: every function returns an int32 status (VBT_OK = 0; 1..9 mirror the VibratoError
 * variants of errors.rs:11-42); out-parameters come last; handles are opaque and released with the
 * matching *_free; vbt_last_error() returns the calling thread's last message (UTF-8, NUL-ended).
 * No torch / CUDA types appear in any signature: device memory is passed as plain addresses.
 *
 * There is NO CPU fallback: functions that run the hot path fail with VBT_ERR_NO_DEVICE /
 * VBT_ERR_CUDA when no usable GPU is present.
 *
 * Threads: a vbt_dict may be shared by readers once built; a vbt_tokenizer owns one workspace and one
 * stream, like a vibrato Worker (tokenizer/worker.rs:14-24), so it serves one caller at a time — create one
 * tokenizer per host thread (they may share the dictionary).  A vbt_result stays valid after its tokenizer is
 * freed.  Inputs are untrusted: dictionary streams, source files and byte offsets are validated, never assumed.
 */
#ifndef VIBRATO_B200_H
#define VIBRATO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    VBT_OK = 0,
    VBT_ERR_INVALID_ARGUMENT = 1, /* VibratoError::InvalidArgument */
    VBT_ERR_INVALID_FORMAT = 2,   /* VibratoError::InvalidFormat   */
    VBT_ERR_TRY_FROM_INT = 3,     /* VibratoError::TryFromInt      */
    VBT_ERR_PARSE_INT = 4,        /* VibratoError::ParseInt        */
    VBT_ERR_DECODE = 5,           /* VibratoError::BincodeDecode   */
    VBT_ERR_ENCODE = 6,           /* VibratoError::BincodeEncode   */
    VBT_ERR_IO = 7,               /* VibratoError::StdIo           */
    VBT_ERR_UTF8 = 8,             /* VibratoError::Utf8            */
    VBT_ERR_UNSUPPORTED = 9,      /* reserved: a recognised input this build cannot run */
    VBT_ERR_CUDA = 100,
    VBT_ERR_NO_DEVICE = 101,
    VBT_ERR_INTERNAL = 102
};

typedef struct vbt_dict vbt_dict;           /* vibrato::Dictionary            (dictionary.rs:54-56) */
typedef struct vbt_tokenizer vbt_tokenizer; /* vibrato::Tokenizer             (tokenizer.rs:13-18)  */
typedef struct vbt_result vbt_result;       /* the top_nodes of a batch of Workers (worker.rs:13-19) */

/* One resultant token: what vibrato::token::Token exposes (token.rs:21-92), sentence-relative.
 * left_id / right_id / word_cost are functions of word_idx: vbt_dict_word_param(). */
typedef struct vbt_token {
    uint32_t start_char; /* Token::range_char().start                     token.rs:21-24 */
    uint32_t end_char;   /* Token::range_char().end                                      */
    uint32_t start_byte; /* Token::range_byte().start                     token.rs:28-32 */
    uint32_t end_byte;   /* Token::range_byte().end                                      */
    uint32_t word_idx;   /* Token::word_idx(): lex_type << 30 | word_id   token.rs:43-46; LexType 0 System,
                            1 User, 2 Unknown (dictionary.rs:30-40) */
    int32_t total_cost;  /* Token::total_cost()                           token.rs:89-92 */
} vbt_token;

/* Opt-in compact record (tokenizer option "compact_tokens" = 1): a third less to bring back over PCIe.  The character
 * range (Token::range_char, token.rs:21-24) is not carried: it is the number of characters of the caller's own UTF-8
 * in front of start_byte / end_byte (sentence.rs:40-46 builds the same table), which the host mirrors rebuild lazily. */
typedef struct vbt_token16 {
    uint32_t start_byte; /* Token::range_byte().start                     token.rs:28-32 */
    uint32_t end_byte;   /* Token::range_byte().end                                      */
    uint32_t word_idx;   /* Token::word_idx()                             token.rs:43-46 */
    int32_t total_cost;  /* Token::total_cost()                           token.rs:89-92 */
} vbt_token16;

#define VBT_WORD_ID(word_idx) ((word_idx) & 0x3FFFFFFFu)
#define VBT_LEX_TYPE(word_idx) ((word_idx) >> 30)

const char *vbt_last_error(void);
/* Library version string, e.g. "vibrato_b200 0.1.0 (sm_100a)". */
const char *vbt_version(void);

/* ---- Dictionary (host) -------------------------------------------------------------------- */

/* Dictionary::read (dictionary.rs:173-197): `dic` is the zstd-DECODED "VibratoTokenizer 0.5\n" stream. */
int32_t vbt_dict_from_bytes(const uint8_t *dic, size_t n, vbt_dict **out);
/* zstd::Decoder::new(File::open(path)) + Dictionary::read, as tokenize/src/main.rs:59-60 does. */
int32_t vbt_dict_from_zstd_file(const char *path, vbt_dict **out);
/* SystemDictionaryBuilder::from_readers (dictionary/builder.rs:64-89): MeCab-format sources. */
int32_t vbt_dict_from_mecab(const char *lex_csv, size_t lex_len, const char *matrix_def, size_t matrix_len,
                            const char *char_def, size_t char_len, const char *unk_def, size_t unk_len,
                            vbt_dict **out);
/* Same with the connection matrix given densely, matrix[left * num_right + right]
 * (MatrixConnector::new, matrix_connector.rs:18-24). */
int32_t vbt_dict_from_parts(const char *lex_csv, size_t lex_len, const int16_t *matrix, uint32_t num_right,
                            uint32_t num_left, const char *char_def, size_t char_len, const char *unk_def,
                            size_t unk_len, vbt_dict **out);
/* SystemDictionaryBuilder::from_readers_with_bigram_info (dictionary/builder.rs:111-148): the connection
 * costs come from bigram.right / bigram.left / bigram.cost through a RawConnector
 * (connector/raw_connector.rs), or with dual_connector != 0 through a DualConnector
 * (connector/dual_connector.rs:155-213; needs >= 8 feature templates, else VBT_ERR_INVALID_ARGUMENT). */
int32_t vbt_dict_from_bigram(const char *lex_csv, size_t lex_len, const char *bigram_right, size_t right_len,
                             const char *bigram_left, size_t left_len, const char *bigram_cost, size_t cost_len,
                             const char *char_def, size_t char_len, const char *unk_def, size_t unk_len,
                             int32_t dual_connector, vbt_dict **out);
/* Test hook for the reference's scorer vectors: ScorerBuilder::insert x n + build + Scorer::accumulate_cost
 * (raw_connector/scorer.rs:110-168, 255-267); triples = n x (key1, key2, cost). */
int32_t vbt_scorer_accumulate(const int32_t *triples, size_t n_triples, const uint32_t *keys1, const uint32_t *keys2,
                              size_t n_keys, int32_t *cost);
/* Dictionary::write (dictionary.rs:142-150). *out is released with vbt_bytes_free. */
int32_t vbt_dict_write(const vbt_dict *d, uint8_t **out, size_t *n);
void vbt_bytes_free(uint8_t *p);
/* Dictionary::reset_user_lexicon_from_reader (dictionary.rs:209-229); csv == NULL clears it. */
int32_t vbt_dict_set_user_lexicon_csv(vbt_dict *d, const char *csv, size_t n);
void vbt_dict_free(vbt_dict *d);

/* Dictionary::word_feature (dictionary.rs:108-114); *p points into the dictionary. */
int32_t vbt_dict_feature(const vbt_dict *d, uint32_t word_idx, const char **p, size_t *len);
/* Dictionary::word_param (dictionary.rs:98-104) -> Token::{left_id,right_id,word_cost} (token.rs:64-85). */
int32_t vbt_dict_word_param(const vbt_dict *d, uint32_t word_idx, uint16_t *left_id, uint16_t *right_id,
                            int16_t *word_cost);
/* Connector::{num_left,num_right} (connector.rs:12-18), lexicon sizes (lex_type 0/1/2). */
int32_t vbt_dict_shape(const vbt_dict *d, uint32_t *num_left, uint32_t *num_right, uint32_t *n_system,
                       uint32_t *n_user, uint32_t *n_unknown);
/* Audit of a lexicon as loaded (lex_type 0 system / 1 user), for dictionaries whose byte layout no reference test
 * pins (tools/validate_dic.py): walks every key of the WordMap's trie (map.rs:33-42, trie.rs:49-56) and looks it up
 * again through the common-prefix search.  out[0] keys, out[1] words (Lexicon::params, lexicon.rs:24-29), out[2]
 * word ids named by the postings of those keys (posting.rs:18-21), out[3] longest key in characters, out[4] keys the
 * search does not find again, out[5] word ids named by no key or by more than one.  A sound lexicon has
 * out[1] == out[2] and out[4] == out[5] == 0. */
int32_t vbt_dict_audit(const vbt_dict *d, int32_t lex_type, uint64_t *out, size_t n_out);
/* Lexicon::common_prefix_iterator (lexicon.rs:33-46) on the host copy: (word_id, end_char) pairs in
 * the order the tokenizer sees them.  *n_out receives the full count even when it exceeds cap. */
int32_t vbt_dict_common_prefix(const vbt_dict *d, int32_t lex_type, const uint32_t *chars, size_t n_chars,
                               uint32_t *word_ids, uint32_t *end_chars, size_t cap, size_t *n_out);

/* Dictionary::map_connection_ids_from_iter (dictionary.rs:245-259): lmap / rmap list the OLD left / right ids in
 * their NEW order (the i-th item, 1-origin, becomes id i; id 0 is reserved), exactly what the `.lmap` / `.rmap`
 * files of the reference's `reorder` tool hold (map/src/main.rs:30-74). */
int32_t vbt_dict_map_connection_ids(vbt_dict *d, const uint16_t *lmap, size_t n_lmap, const uint16_t *rmap,
                                    size_t n_rmap);
/* ConnectorCost::cost (matrix_connector.rs:121-124) and CharProperty::char_info (character.rs:112-116, the
 * packed CharInfo of character.rs:10-24) on the host copy. */
int32_t vbt_dict_conn_cost(const vbt_dict *d, uint16_t right_id, uint16_t left_id, int32_t *cost);
int32_t vbt_dict_char_info(const vbt_dict *d, uint32_t code_point, uint32_t *char_info);
/* CharProperty::cate_id (character.rs:119-124): *id = -1 when the category is not defined. */
int32_t vbt_dict_cate_id(const vbt_dict *d, const char *name, size_t len, int32_t *id);

/* The packed device image of the dictionary (see vibrato_b200/csrc/device_blob.hpp).  Rank 0 packs
 * and uploads it; other ranks receive the same bytes over NCCL and hand the device address to
 * vbt_tokenizer_new_from_device_blob. */
int32_t vbt_dict_blob_size(const vbt_dict *d, uint64_t *n_bytes);
int32_t vbt_dict_pack_blob(const vbt_dict *d, uint8_t *host_dst, uint64_t n_bytes);

/* ---- Tokenizer (device) ------------------------------------------------------------------- */

/* Tokenizer::new(dict).ignore_space(ignore_space)?.max_grouping_len(max_grouping_len)
 * (tokenizer.rs:26-74): uploads the dictionary image to `device` (a CUDA ordinal).
 * Fails with VBT_ERR_INVALID_ARGUMENT when ignore_space is set and char.def has no SPACE
 * category (tokenizer.rs:44-49).  max_grouping_len == 0 means unlimited (tokenizer.rs:67-74). */
int32_t vbt_tokenizer_new(const vbt_dict *d, int32_t ignore_space, uint64_t max_grouping_len, int32_t device,
                          vbt_tokenizer **out);
/* Same, over a dictionary image that already sits in `device`'s memory at d_blob (n_bytes long;
 * e.g. the receive buffer of an NCCL broadcast).  The tokenizer does not take ownership. */
int32_t vbt_tokenizer_new_from_device_blob(uint64_t d_blob, uint64_t n_bytes, int32_t ignore_space,
                                           uint64_t max_grouping_len, int32_t device, vbt_tokenizer **out);
/* One tokenizer over `n_devices` GPUs of this node (SURVEY.md §8(b)-3/4, §8(e); no reference counterpart: a vibrato
 * Worker is one CPU thread, worker.rs:13-31 — the contract is BASELINE.json's north_star).  The dictionary image is
 * uploaded once, to devices[0], and broadcast to the others (ncclBroadcast when libnccl.so.2 can be loaded, peer
 * copies otherwise).  vbt_tokenize_batch cuts the batch into contiguous shards of about equal bytes, runs one
 * engine per device on its own host thread (pinned to the GPU's NUMA node) and returns ONE result in input order,
 * identical to a single-device one.  vbt_tokenize_batch_device expects its input on devices[0] and gathers the
 * token records back to it over NVLink (ncclSend / ncclRecv).  Not available on such a tokenizer: a caller-owned
 * stream and the output stage ("output_mode"). */
int32_t vbt_tokenizer_new_multi(const vbt_dict *d, int32_t ignore_space, uint64_t max_grouping_len,
                                const int32_t *devices, int32_t n_devices, vbt_tokenizer **out);
/* JSON description of how the tokenizer is laid out: {"devices": [...], "dictionary_transport": "nccl 22703" |
 * "cudaMemcpyPeer" | "single device", "token_gather": ..., "numa_pinned": [...]}. */
int32_t vbt_tokenizer_describe(const vbt_tokenizer *t, char *buf, size_t cap);
/* Restricts the calling thread to the CPUs of the NUMA node `device` hangs off (host-side copies of a rank then
 * stay on its socket); never widens the process's own affinity mask. */
int32_t vbt_pin_thread_to_device(int32_t device);
void vbt_tokenizer_free(vbt_tokenizer *t);

/* for each sentence: Worker::reset_sentence + Worker::tokenize (worker.rs:34-55), batched.
 * Sentence i is utf8[byte_offsets[i] .. byte_offsets[i+1]) and must be valid UTF-8 (else
 * VBT_ERR_UTF8, the failure `stdin.lines()` reports at tokenize/src/main.rs:79).  HOST pointers:
 * the call copies the input to the device, runs the kernels and copies the tokens back.
 * An empty sentence yields zero tokens (worker.rs:50-52). */
int32_t vbt_tokenize_batch(vbt_tokenizer *t, const char *utf8, const uint64_t *byte_offsets, uint64_t n_sent,
                           vbt_result **out);
/* Worker::num_tokens / token(i) / token_iter (worker.rs:59-74) for the whole batch:
 * tokens of sentence i are toks[tok_offsets[i] .. tok_offsets[i+1]), in sentence order. */
int32_t vbt_result_view(const vbt_result *r, const uint64_t **tok_offsets, const vbt_token **toks,
                        uint64_t *n_sent, uint64_t *n_tokens);
/* The same for a batch tokenised with the option "compact_tokens" = 1 (vbt_result_view refuses such a result and this
 * call refuses a full one).  With that option vbt_tokenize_batch_device's d_tokens are vbt_token16 records too. */
int32_t vbt_result_view_compact(const vbt_result *r, const uint64_t **tok_offsets, const vbt_token16 **toks,
                                uint64_t *n_sent, uint64_t *n_tokens);
/* The output loop of `tokenize` (tokenize/src/main.rs:83-127) for the whole batch, formatted on the device when the
 * tokenizer option "output_mode" was 1 (mecab: `surface\tfeature\n`.. `EOS\n`), 2 (wakati: surfaces joined by ' ',
 * `\n`) or 3 (detail: mecab + lex_type/left_id/right_id/word_cost/total_cost) during vbt_tokenize_batch: sentence i's
 * lines are text[text_offsets[i] .. text_offsets[i+1]).  VBT_ERR_INVALID_ARGUMENT when the option was off. */
int32_t vbt_result_text(const vbt_result *r, const uint64_t **text_offsets, const char **text, uint64_t *n_bytes);
/* The loop of the `evaluate` tool (evaluate/src/main.rs:61-138): corpus = `surface\tfeature` lines with `EOS`
 * between sentences (Corpus::from_reader, trainer/corpus.rs:78-121); every sentence (its surfaces concatenated) is
 * tokenised in one batch and compared with the corpus as sets of (char range, features[feature_indices]) — all
 * features when n_indices == 0, "*" for a missing index.  Precision = num_cor / num_sys, recall = num_cor / num_ref.
 * `d` must be the dictionary `t` was created from. */
int32_t vbt_evaluate(const vbt_dict *d, vbt_tokenizer *t, const char *corpus, size_t len, const uint64_t *feature_indices,
                     size_t n_indices, uint64_t *num_ref, uint64_t *num_sys, uint64_t *num_cor);
void vbt_result_free(vbt_result *r);

/* Device-resident variant: d_utf8 / d_byte_offsets are DEVICE addresses of the same two arrays
 * (n_bytes = byte_offsets[n_sent]); results stay in device memory owned by the tokenizer and are
 * valid until its next call: *d_tok_offsets -> uint64[n_sent+1], *d_tokens -> vbt_token[*n_tokens]. */
int32_t vbt_tokenize_batch_device(vbt_tokenizer *t, uint64_t d_utf8, uint64_t d_byte_offsets, uint64_t n_sent,
                                  uint64_t n_bytes, uint64_t *d_tok_offsets, uint64_t *d_tokens,
                                  uint64_t *n_tokens);

/* Pinned host memory for callers that want full-speed host<->device copies. */
int32_t vbt_host_alloc(size_t n_bytes, void **out);
void vbt_host_free(void *p);

/* Measurement hooks (bench.py): per-stage device time of the last batch in milliseconds, in the
 * order reported by vbt_stage_names(); number of kernels the last batch launched; and the
 * algorithmic-byte counters U,C,M,T,P,W,E,N,K of SURVEY.md §8(d) measured on the device. */
/* Turns the device-side counters on or off (off by default: they cost an extra walk per position). */
int32_t vbt_tokenizer_set_counting(vbt_tokenizer *t, int32_t on);
/* Tuning knobs (results never change): "chunk_sentences" = sentences per chunk of the pipelined host path
 * (default 262144, 0 = off), "counting" = 0|1, "connid_counting" = 0|1 (see vbt_connid_counts),
 * "output_mode" = 0|1|2|3 (see vbt_result_text; default 0). */
int32_t vbt_tokenizer_set_option(vbt_tokenizer *t, const char *name, int64_t value);
/* Worker::init_connid_counter / update_connid_counts / compute_connid_probs (worker.rs:77-103): switch
 * the option "connid_counting" on (this zeroes the counters), tokenise the corpus, then read the edge
 * counts of every lattice (Lattice::add_connid_counts, lattice.rs:170-183) in the dictionary's own ids:
 * lid_count[num_left], rid_count[num_right].  Pass NULL arrays to query the sizes only. */
int32_t vbt_connid_counts(vbt_tokenizer *t, uint64_t *lid_count, uint64_t *rid_count, uint32_t *num_left,
                          uint32_t *num_right);
/* Launch the kernels on a caller-owned CUDA stream (a cudaStream_t passed as an integer; 0 restores
 * the tokenizer's own stream), so callers can bracket batches with their own events. */
int32_t vbt_tokenizer_set_stream(vbt_tokenizer *t, uint64_t stream);
int32_t vbt_last_stage_ms(const vbt_tokenizer *t, float *ms, int32_t cap, int32_t *n_stages);
const char *vbt_stage_names(void);
int32_t vbt_last_launch_count(const vbt_tokenizer *t, uint64_t *n_launches);
/* cnt10 = U,C,M,T,P,W,E,N,K,walks of the last batch run with counting on. */
int32_t vbt_last_counters(const vbt_tokenizer *t, uint64_t *cnt10);

#ifdef __cplusplus
}
#endif
#endif
