// Device-side views and kernel declarations of the batched Viterbi tokenizer (sm_100a).
//
// Flattened "slot" space: sentence s with n_s characters owns slots [slot_off[s], slot_off[s]+n_s];
// the last one is a sentinel standing for character position n_s (the `ends[len]` row of
// vibrato's Lattice, tokenizer/lattice.rs:38-43).  All per-character arrays are indexed by slot.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace vbt {

struct DictView {
    const uint32_t* chr2inf;
    uint32_t chr2inf_len;
    const uint32_t* sys_table;
    uint32_t sys_table_len;
    const uint4* sys_nodes;  // {base, check, postings index of the key ending here or kNone, its word count}
    uint32_t sys_num_nodes;
    const uint4* sys_post;  // per key {len,0,0,0} then len candidate records {left|right<<16, cost word, word_idx, 0}
    const uint32_t* usr_table;  // nullptr when there is no user lexicon
    uint32_t usr_table_len;
    const uint4* usr_nodes;
    uint32_t usr_num_nodes;
    const uint4* usr_post;
    const uint32_t* unk_off;
    const uint2* unk_ent;  // {left | right << 16, cost}
    const int16_t* matrix;  // connector_kind 0 (MatrixConnector); the reduced matrix of connector_kind 2
    uint32_t num_right;     // row length of the reduced matrix (connector_kind 2)
    uint32_t conn_stride_left, conn_stride_right;  // connector_kind 0: cost = matrix[left * sl + right * sr]
    uint32_t opaque_zero;    // always 0; a value the compiler cannot fold (k_viterbi2 uses it to order its loads)
    uint32_t matrix_window;  // connector_kind 0: 1 = the matrix does not cross a 4 GiB address boundary (k_viterbi2)
    // connector_kind 1 (RawConnector, connector/raw_connector.rs + raw_connector/scorer.rs)
    uint32_t connector_kind;
    const uint32_t* right_feats;  // [num_right][feat_T]
    const uint32_t* left_feats;   // [num_left][feat_T]
    uint32_t feat_T;
    const uint32_t* sc_bases;
    const uint32_t* sc_checks;
    const int32_t* sc_costs;
    uint32_t n_bases, n_checks;
    // connector_kind 2 (DualConnector, connector/dual_connector.rs): connection id -> column / row of `matrix`,
    // plus the raw fields above with feat_T == 8
    const uint16_t* right_conn;
    const uint16_t* left_conn;
    // output stage: per lexicon type (0 system, 1 user, 2 unknown) features and dictionary-id parameters by word id
    const uint32_t* feat_off[3];
    const uint8_t* feat[3];
    const uint2* params[3];  // {left | right << 16, word_cost (i16, sign-extended in the low half)}
    uint32_t n_words[3];
    uint32_t space_mask;         // 1 << cate_id("SPACE") when ignore_space, else 0 (tokenizer.rs:16,42-55)
    unsigned long long max_grouping;  // ~0ull when unlimited (tokenizer.rs:17,67-74)
};

enum : uint32_t {
    kFlagUtf8Error = 1u,
    kFlagPoolOverflow = 2u,
    kFlagBadOffsets = 4u,  // byte_off decreases or leaves the input buffer
    // some sentence is so long that path costs may leave +-2^30: k_viterbi2 then runs without its lower-bound
    // pruning, whose arithmetic assumes that no i32 addition wraps
    kFlagLongSentence = 8u,
    // the batch has more characters than the per-character kernels were launched for (the engine sizes those
    // launches from a learned characters-per-byte ratio): later kernels stand down, the engine re-runs the batch
    kFlagSlotsOverflow = 16u,
};
constexpr uint32_t kFlagsStandDown = kFlagBadOffsets | kFlagSlotsOverflow;
constexpr uint32_t kPruneMaxChars = 16000;  // (chars + 1) nodes x 65 535 per node < 2^30

enum : uint32_t { kInfoTrailing = 1u };  // tokenizer.rs:128-130: the input ends with skipped spaces
constexpr uint32_t kInfoSpecial = 0x80000000u;  // Batch::info[slot].y: info_ex[slot] holds a skip or a flag

constexpr uint32_t kInvalidCode = 0xFFFFFFFFu;
constexpr uint32_t kNone = 0xFFFFFFFFu;

// Counter slots (SURVEY.md §8d) inside Batch::counters
enum { kCntU = 0, kCntC, kCntM, kCntT, kCntP, kCntW, kCntE, kCntN, kCntK, kCntWalks, kNumCounters };

struct Batch {
    // input
    const uint8_t* utf8;
    const unsigned long long* byte_off;  // n_sent + 1
    unsigned long long total_bytes;      // size of the buffer behind utf8: no offset may exceed it
    uint32_t n_sent;
    uint32_t launch_slots;  // slots the per-character launches (K2, the row-offset scan) cover
    // per sentence
    uint32_t* n_slots;   // chars + 1 (scan input)
    uint32_t* slot_off;  // n_sent + 1
    uint4* eos;          // {best prev entry, start_node (sentence-relative), cost, 0}
    uint32_t* n_tok;
    unsigned long long* tok_off;  // n_sent + 1
    // per slot
    uint32_t* code_sys;
    uint32_t* code_usr;
    uint32_t* cinfo;
    uint32_t* groupable;  // 0 marks the sentinel slot
    uint32_t* byte_pos;   // byte offset of the character inside its sentence (c2b, sentence.rs:40-46)
    uint2* info;          // {cand_ptr, cand_cnt | kInfoSpecial}
    uint2* info_ex;       // {skip (start_word - start_node), flags}; written only where info.y has kInfoSpecial
    uint32_t* ends_cnt;   // upper bound of nodes ending here (+1 for BOS at the first slot)
    uint2* ends_meta;     // {exclusive scan of ends_cnt = row offset, next free entry of the row (absolute index)}
    // candidate pool and lattice rows
    // {left | right << 16, word_cost (i16, low half) | lower bound of the connection cost into `left` (i16, high
    //  half; see device_blob.hpp), word_idx, end_slot}
    uint4* cand;
    uint32_t cand_cap;
    int2* ends_hot;       // lattice rows (CSR over end slot): {min_cost, right_id} — all the DP re-reads
    uint4* ends_cold;     // {start_node slot, best prev entry, word_idx, min_cost} — written once, read by the backtrack
    // output
    void* tokens;  // vbt_token[] (24 bytes each), or vbt_token16[] when compact != 0
    uint32_t compact;  // 1: 16-byte records {start_byte, end_byte, word_idx, total_cost} (character ranges left to the host)
    // bookkeeping
    unsigned long long* pool_ctr;
    uint32_t* flags;
    unsigned long long* counters;  // kNumCounters, or nullptr when counting is off
    // ConnIdCounter (mapper.rs:87-104) over internal ids, or nullptr: lid_count[num_left], rid_count[num_right]
    unsigned long long* lid_count;
    unsigned long long* rid_count;
};

// Output stage: what `tokenize` prints per sentence (tokenize/src/main.rs:83-127), produced on the device.
enum : uint32_t { kOutNone = 0, kOutMecab = 1, kOutWakati = 2, kOutDetail = 3 };
struct FormatArgs {
    const uint8_t* utf8;
    const unsigned long long* byte_off;  // n_sent + 1
    uint32_t n_sent;
    const unsigned long long* tok_off;   // n_sent + 1
    const uint2* tokens;                 // vbt_token as 3 x uint2
    uint32_t* tok_len;                   // bytes each token contributes (separators included, terminators not)
    const unsigned long long* tok_text_off;  // exclusive scan of tok_len, n_tokens + 1
    unsigned long long* text_off;        // n_sent + 1: where each sentence's text starts
    uint8_t* text;
    uint32_t mode;
};
void launch_format_len(const DictView& d, const FormatArgs& f, cudaStream_t st);
void launch_format_write(const DictView& d, const FormatArgs& f, cudaStream_t st);

void launch_count_chars(const Batch& b, cudaStream_t st);
void launch_decode(const DictView& d, const Batch& b, cudaStream_t st);
void launch_candidates(const DictView& d, const Batch& b, uint32_t max_slots, cudaStream_t st);
// K3 = k_viterbi2.  kernel (matrix connector only): 1 = lower-bound pruning, with its unpruned twin for batches with
// very long sentences; 0 = the unpruned 64-bit-address lookup that a matrix crossing a 4 GiB address boundary takes
// anyway.  Returns the number of kernels launched.
int launch_viterbi(const DictView& d, const Batch& b, int kernel, cudaStream_t st);
// Counted runs only (b.counters or b.lid_count): the SURVEY.md §8(d) counters M, T, P, W, walks, E, N and the
// connection-id counts, read off the lattice K3 left.  Runs between K3 and launch_backtrack_count.
void launch_count_lattice(const DictView& d, const Batch& b, cudaStream_t st);
void launch_backtrack_count(const Batch& b, cudaStream_t st);
void launch_backtrack_write(const Batch& b, cudaStream_t st);

}  // namespace vbt
