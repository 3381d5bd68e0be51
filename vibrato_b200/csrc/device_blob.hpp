// One contiguous, position-independent image of everything the kernels read from the dictionary.
// Built once on the host (pack_device_blob), copied to HBM once (or NCCL-broadcast between ranks)
// and viewed through offsets in the header, so the same bytes work on every GPU.
//
// HBM layout (every section 256-byte aligned so rows/sections can be fetched with bulk copies):
//
//   BlobHeader                                   512 B
//   chr2inf      u32[chr2inf_len]                character.rs:105-116 (CharInfo table)
//   sys_table    u32[sys_table_len]              code point -> trie code (crawdad CodeMapper)
//   sys_nodes    {u32 base, u32 check, u32 value, u32 len}[n]   double array (crawdad semantics) + per node the
//                                                device postings index and word count of the key ending there
//   sys_post     uint4[...]                      per key: {len,0,0,0}, then len x {left|right<<16, cost word, word_idx, 0}
//                                                cost word = word_cost (i16, low half) | lb << 16, lb = min over all right
//                                                ids of MatrixConnector::cost(right, left) (INT16_MIN for Raw / Dual)
//   usr_table / usr_nodes / usr_post             same for the user lexicon (absent when none)
//   unk_off      u32[n_categories + 1]           unknown.rs:63-66
//   unk_ent      {u32 left|right<<16, u32 cost word}[n_unk]
//   matrix       i16[num_right][num_left]        matrix_connector.rs:11-15 transposed: cost = m[right*num_left+left]
//   left_ids / right_ids u16[]                    internal connection id -> dictionary connection id
//   Raw connector instead of matrix:              right_feats u32[num_right][feat_T], left_feats u32[num_left][feat_T],
//                                                 bases u32[], checks u32[], costs i32[]   (raw_connector.rs, scorer.rs)
//   feat_off / feat / params x {sys, usr, unk}    feature strings and {left, right, cost} per word id, for the
//                                                 device-side output stage (k_format_*)
//   Dual connector (dual_connector.rs):           reduced matrix i16[m_num_left][m_num_right] in `matrix`, the raw
//                                                 sections with feat_T = 8, right_conn u16[num_right], left_conn u16[num_left]
//
// Connection ids inside the image (postings, unk entries, matrix rows/columns) are renumbered by
// descending usage estimate with id 0 fixed (see pack_device_blob); no API exposes them.
#pragma once

#include <cstdint>
#include <vector>

#include "host_dict.hpp"

namespace vbt {

constexpr uint64_t kBlobMagic = 0x3430424F4C425456ull;  // "VTBLOB04"

struct BlobHeader {
    uint64_t magic;
    uint64_t total_bytes;
    uint32_t num_right, num_left;
    uint32_t chr2inf_len;
    uint32_t n_categories;
    int32_t space_cate_id;  // -1 when char.def defines no SPACE (tokenizer.rs:44-49)
    uint32_t has_user;
    uint32_t sys_table_len, sys_num_nodes, sys_post_len;
    uint32_t usr_table_len, usr_num_nodes, usr_post_len;
    uint32_t n_unk;
    uint32_t reserved0;
    uint64_t off_chr2inf, off_sys_table, off_sys_nodes, off_sys_post;
    uint64_t off_usr_table, off_usr_nodes, off_usr_post;
    uint64_t off_unk_off, off_unk_ent, off_matrix;
    uint64_t off_left_ids, off_right_ids;  // u16[num_left] / u16[num_right]: internal id -> dictionary id
    // Raw connector (connector_kind == 1): feature rows and the scorer's double array; off_matrix is unused
    uint32_t connector_kind, feat_T, n_bases, n_checks;
    uint64_t off_right_feats, off_left_feats, off_bases, off_checks, off_costs;
    // Dual connector (connector_kind == 2): off_matrix holds the reduced matrix i16[m_num_left][m_num_right],
    // these map an internal connection id to its column/row of it, and the raw sections hold the 8-lane term
    uint64_t off_right_conn, off_left_conn;  // u16[num_right] / u16[num_left]
    uint32_t m_num_right, m_num_left;
    uint32_t matrix_transposed;  // connector_kind 0: always 1, the matrix is i16[num_right][num_left]; the engine
                                 // refuses an image with any other value
    uint32_t reserved1;
    // Output stage (tokenize/src/main.rs:83-127): per lexicon (0 system, 1 user, 2 unknown) the feature strings
    // (feat_off u32[n_words + 1] into feat bytes) and the word parameters in the dictionary's own connection
    // ids ({left u16, right u16, cost i16, 0}: Token::{left_id,right_id,word_cost}, token.rs:64-85)
    uint32_t n_words[3];
    uint32_t reserved2;
    uint64_t off_feat_off[3], off_feat[3], off_params[3];
    uint8_t pad[512 - 8 * 2 - 4 * 14 - 8 * 12 - 4 * 4 - 8 * 5 - 8 * 2 - 4 * 2 - 4 * 2 - 4 * 4 - 8 * 9];
};
static_assert(sizeof(BlobHeader) == 512, "BlobHeader must stay 512 bytes");

// Validates every index the kernels will trust (trie leaf values, postings ids, unk offsets,
// connection ids) and throws vbt::Error otherwise.
void pack_device_blob(const Dictionary& d, std::vector<uint8_t>& out);

}  // namespace vbt
