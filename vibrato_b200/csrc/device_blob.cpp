#include "device_blob.hpp"

#include <algorithm>
#include <cstring>
#include <thread>

namespace vbt {

namespace {

uint64_t align256(uint64_t x) { return (x + 255) & ~uint64_t(255); }

struct LexSizes {
    uint64_t table_bytes, nodes_bytes, post_bytes;
    std::vector<uint32_t> post_map;  // host postings offset -> device postings index in 16-byte units (or ~0u)
    uint32_t post_len;
};

LexSizes measure(const Lexicon& lx) {
    LexSizes s;
    s.table_bytes = uint64_t(lx.trie.table.size()) * 4;
    s.nodes_bytes = uint64_t(lx.trie.num_nodes()) * 16;
    s.post_map.assign(lx.postings.size(), 0xFFFFFFFFu);
    uint64_t dev = 0;
    for (size_t i = 0; i < lx.postings.size();) {
        uint64_t len = lx.postings[i];
        if (i + 1 + len > lx.postings.size()) throw Error(kDecode, "postings overrun");
        if (dev > 0x7FFFFFFFull) throw Error(kTryFromInt, "postings too large for the device layout");
        s.post_map[i] = uint32_t(dev);
        dev += 1 + len;  // in 16-byte units: one header, one record per word
        i += 1 + len;
    }
    if (dev > 0x7FFFFFFFull) throw Error(kTryFromInt, "postings too large for the device layout");
    s.post_len = uint32_t(dev);
    s.post_bytes = dev * 16;
    return s;
}

// Cost word of a candidate: the i16 word cost in the low half, the lower bound of every connection cost into the
// word's left id in the high half (k_viterbi2's pruning; INT16_MIN where no bound is known).
inline uint32_t pack_cost(int16_t word_cost, int16_t conn_lower_bound) {
    return uint32_t(uint16_t(word_cost)) | (uint32_t(uint16_t(conn_lower_bound)) << 16);
}

void write_lexicon(const Lexicon& lx, const LexSizes& s, const std::vector<uint16_t>& lmap,
                   const std::vector<uint16_t>& rmap, const std::vector<int16_t>& left_lb, uint8_t* table,
                   uint8_t* nodes, uint8_t* post) {
    if (!lx.trie.table.empty()) std::memcpy(table, lx.trie.table.data(), s.table_bytes);
    // Device node = {base, check, value, len}: crawdad's base / check (trie.rs:14-27 semantics: MSB(base) = leaf,
    // MSB(check) = a key ends here) plus, where a key ends at the node, the device postings index of that key and
    // the number of words it lists — so that a step of the walk is ONE 16-byte load and a hit needs neither the
    // fetch of the terminal child nor of the postings header (two dependent loads less per hit than the blob's
    // own layout).
    uint32_t nn = lx.trie.num_nodes();
    uint32_t* dn = reinterpret_cast<uint32_t*>(nodes);
    auto device_value = [&](uint32_t v, uint32_t* len) {
        if (v >= s.post_map.size() || s.post_map[v] == 0xFFFFFFFFu)
            throw Error(kDecode, "trie value does not point at a postings list");
        *len = lx.postings[v];
        return s.post_map[v];
    };
    for (uint32_t i = 0; i < nn; ++i) {
        uint32_t b = lx.trie.nodes[2 * size_t(i)], c = lx.trie.nodes[2 * size_t(i) + 1];
        uint32_t value = 0xFFFFFFFFu, len = 0;
        bool vacant = (b == Trie::kMask && c == Trie::kMask);
        if (!vacant) {
            if (b & Trie::kFlag) {  // leaf: the value is an offset into Postings.data (map.rs:63-66)
                value = device_value(b & Trie::kMask, &len);
            } else if (c & Trie::kFlag) {
                // has_leaf: the terminal child sits at base ^ 0; it must be a leaf owned by this node
                const uint32_t t = b & Trie::kMask;
                if (t >= nn || !(lx.trie.nodes[2 * size_t(t)] & Trie::kFlag) ||
                    (lx.trie.nodes[2 * size_t(t) + 1] & Trie::kMask) != i)
                    throw Error(kDecode, "trie node flags a terminal child that is not its leaf");
                value = device_value(lx.trie.nodes[2 * size_t(t)] & Trie::kMask, &len);
            }
        }
        dn[4 * size_t(i)] = b;
        dn[4 * size_t(i) + 1] = c;
        dn[4 * size_t(i) + 2] = value;
        dn[4 * size_t(i) + 3] = len;
    }
    // 16-byte records: per key a header {len, 0, 0, 0}, then per word the candidate record k_candidates copies
    // as is, {left | right << 16, cost word, word_idx, 0 (end slot, filled in by the kernel)}
    uint32_t* dp = reinterpret_cast<uint32_t*>(post);
    size_t o = 0;
    for (size_t i = 0; i < lx.postings.size();) {
        uint32_t len = lx.postings[i];
        dp[o++] = len;
        dp[o++] = 0;
        dp[o++] = 0;
        dp[o++] = 0;
        for (uint32_t k = 0; k < len; ++k) {
            uint32_t wid = lx.postings[i + 1 + k];
            if (wid >= lx.params.size()) throw Error(kDecode, "postings word id out of range");
            const WordParam& p = lx.params[wid];
            dp[o++] = uint32_t(lmap[p.left_id]) | (uint32_t(rmap[p.right_id]) << 16);
            dp[o++] = pack_cost(p.word_cost, left_lb[p.left_id]);
            dp[o++] = pack_word_idx(lx.lex_type, wid);
            dp[o++] = 0;
        }
        i += 1 + len;
    }
}

}  // namespace

void pack_device_blob(const Dictionary& d, std::vector<uint8_t>& out) {
    if (d.connector_kind != kMatrix && d.connector_kind != kRaw && d.connector_kind != kDual)
        throw Error(kUnsupported, "unknown connector kind");
    const bool dual = d.connector_kind == kDual;
    const bool raw = d.connector_kind != kMatrix;  // raw sections present (Raw, and the 8-lane term of Dual)
    const bool has_matrix = d.connector_kind != kRaw;
    const uint32_t nl = d.num_left(), nr = d.num_right();
    if (nl == 0 || nr == 0) throw Error(kDecode, "empty connector");
    if (has_matrix && d.matrix.data.size() != size_t(d.matrix.num_left) * d.matrix.num_right)
        throw Error(kDecode, "matrix shape mismatch");
    if (has_matrix && d.matrix.data.size() > 0xFFFFFFFFull)  // the kernels index the matrix with 32 bits
        throw Error(kUnsupported, "connection matrix with 2^32 or more entries (8 GiB) does not fit the device image");
    if (dual) {
        if (d.raw.feat_T != 8 || d.dual_left_map.size() != nl || d.dual_right_map.size() != nr)
            throw Error(kDecode, "dual connector shape mismatch");
        for (uint16_t v : d.dual_right_map)
            if (v >= d.matrix.num_right) throw Error(kDecode, "dual connector: right id map leaves the matrix");
        for (uint16_t v : d.dual_left_map)
            if (v >= d.matrix.num_left) throw Error(kDecode, "dual connector: left id map leaves the matrix");
    }
    if (raw && (d.raw.right_feats.size() != size_t(nr) * d.raw.feat_T || d.raw.left_feats.size() != size_t(nl) * d.raw.feat_T ||
                d.raw.checks.size() != d.raw.costs.size()))
        throw Error(kDecode, "raw connector shape mismatch");
    if (!d.system.verify(nl, nr) || !d.unk.verify(nl, nr) || (d.user && !d.user->verify(nl, nr)))
        throw Error(kInvalidArgument, "connection ids outside the matrix");
    if (d.char_prop.chr2inf.empty()) throw Error(kDecode, "empty chr2inf");
    const uint32_t n_cat = uint32_t(d.unk.offsets.size() ? d.unk.offsets.size() - 1 : 0);
    for (uint32_t ci : d.char_prop.chr2inf)
        if (((ci >> 18) & 0xFF) >= n_cat) throw Error(kDecode, "CharInfo base_id has no unk.def slot");
    for (size_t i = 0; i + 1 < d.unk.offsets.size(); ++i)
        if (d.unk.offsets[i] > d.unk.offsets[i + 1] || d.unk.offsets[i + 1] > d.unk.entries.size())
            throw Error(kDecode, "unk offsets out of range");

    LexSizes ss = measure(d.system), us{};
    if (d.user) us = measure(*d.user);

    // Device-internal connection-id order: ids sorted by how many dictionary entries carry them, id 0
    // (BOS/EOS) fixed.  Tokens never expose connection ids (only word_idx), so this is invisible to
    // callers; it clusters the frequently used rows/columns of the matrix so that they stay
    // L2-resident — the effect vibrato's offline `reorder`/`map` tools go after (docs/map.md,
    // mapper.rs:87-146), applied here at image-pack time with a static usage estimate.
    std::vector<uint16_t> lmap, rmap;
    {
        std::vector<uint64_t> lc(nl, 0), rc(nr, 0);
        auto tally = [&](const Lexicon& lx) {
            for (auto& p : lx.params) {
                ++lc[p.left_id];
                ++rc[p.right_id];
            }
        };
        tally(d.system);
        if (d.user) tally(*d.user);
        for (auto& e : d.unk.entries) {
            lc[e.left_id] += 4;
            rc[e.right_id] += 4;
        }
        auto order_of = [](const std::vector<uint64_t>& cnt) {
            std::vector<uint32_t> idx(cnt.size());
            for (uint32_t i = 0; i < idx.size(); ++i) idx[i] = i;
            std::stable_sort(idx.begin() + 1, idx.end(), [&](uint32_t a, uint32_t b) { return cnt[a] > cnt[b]; });
            std::vector<uint16_t> map(cnt.size());
            for (uint32_t n = 0; n < idx.size(); ++n) map[idx[n]] = uint16_t(n);
            return map;
        };
        lmap = order_of(lc);
        rmap = order_of(rc);
    }

    // Lower bound of MatrixConnector::cost(right, left) over all right ids, per (dictionary) left id.
    std::vector<int16_t> left_lb(nl, INT16_MIN);
    if (d.connector_kind == kMatrix) {
        const int16_t* m = d.matrix.data.data();
        for (uint32_t l = 0; l < nl; ++l) {
            const int16_t* row = m + size_t(l) * nr;
            int16_t lo = row[0];
            for (uint32_t r = 1; r < nr; ++r) lo = std::min(lo, row[r]);
            left_lb[l] = lo;
        }
    }

    BlobHeader h;
    std::memset(&h, 0, sizeof(h));
    h.magic = kBlobMagic;
    h.num_right = nr;
    h.num_left = nl;
    h.chr2inf_len = uint32_t(d.char_prop.chr2inf.size());
    h.n_categories = n_cat;
    h.space_cate_id = d.char_prop.cate_id("SPACE");
    h.has_user = d.user ? 1 : 0;
    h.sys_table_len = uint32_t(d.system.trie.table.size());
    h.sys_num_nodes = d.system.trie.num_nodes();
    h.sys_post_len = ss.post_len;
    if (d.user) {
        h.usr_table_len = uint32_t(d.user->trie.table.size());
        h.usr_num_nodes = d.user->trie.num_nodes();
        h.usr_post_len = us.post_len;
    }
    h.n_unk = uint32_t(d.unk.entries.size());
    uint64_t off = sizeof(BlobHeader);
    auto place = [&](uint64_t bytes) {
        uint64_t o = off;
        off = align256(off + bytes);
        return o;
    };
    h.off_chr2inf = place(uint64_t(h.chr2inf_len) * 4);
    h.off_sys_table = place(ss.table_bytes);
    h.off_sys_nodes = place(ss.nodes_bytes);
    h.off_sys_post = place(ss.post_bytes);
    h.off_usr_table = place(us.table_bytes);
    h.off_usr_nodes = place(us.nodes_bytes);
    h.off_usr_post = place(us.post_bytes);
    h.off_unk_off = place(uint64_t(n_cat + 1) * 4);
    h.off_unk_ent = place(uint64_t(h.n_unk) * 8);
    h.off_matrix = place(has_matrix ? uint64_t(d.matrix.data.size()) * 2 : 0);
    h.connector_kind = uint32_t(d.connector_kind);
    h.m_num_right = has_matrix ? d.matrix.num_right : 0;
    h.m_num_left = has_matrix ? d.matrix.num_left : 0;
    if (dual) {
        h.off_right_conn = place(uint64_t(nr) * 2);
        h.off_left_conn = place(uint64_t(nl) * 2);
    }
    if (raw) {
        h.feat_T = d.raw.feat_T;
        h.n_bases = uint32_t(d.raw.bases.size());
        h.n_checks = uint32_t(d.raw.checks.size());
        h.off_right_feats = place(d.raw.right_feats.size() * 4);
        h.off_left_feats = place(d.raw.left_feats.size() * 4);
        h.off_bases = place(d.raw.bases.size() * 4);
        h.off_checks = place(d.raw.checks.size() * 4);
        h.off_costs = place(d.raw.costs.size() * 4);
    }
    h.off_left_ids = place(uint64_t(nl) * 2);
    h.off_right_ids = place(uint64_t(nr) * 2);
    // output stage: features and parameters by word id
    uint64_t unk_feat_bytes = 0;
    for (auto& e : d.unk.entries) unk_feat_bytes += e.feature.size();
    const Lexicon* lexs[2] = {&d.system, d.user ? &*d.user : nullptr};
    for (int li = 0; li < 3; ++li) {
        const uint64_t nw = li < 2 ? (lexs[li] ? lexs[li]->num_words() : 0) : d.unk.entries.size();
        const uint64_t fb = li < 2 ? (lexs[li] ? lexs[li]->feature_blob.size() : 0) : unk_feat_bytes;
        if (fb > 0xFFFFFFFFull) throw Error(kTryFromInt, "feature strings too large for the device layout");
        h.n_words[li] = uint32_t(nw);
        h.off_feat_off[li] = place((nw + 1) * 4);
        h.off_feat[li] = place(fb);
        h.off_params[li] = place(nw * 8);
    }
    h.total_bytes = off;

    out.assign(off, 0);
    std::memcpy(out.data(), &h, sizeof(h));
    std::memcpy(out.data() + h.off_chr2inf, d.char_prop.chr2inf.data(), size_t(h.chr2inf_len) * 4);
    write_lexicon(d.system, ss, lmap, rmap, left_lb, out.data() + h.off_sys_table, out.data() + h.off_sys_nodes,
                  out.data() + h.off_sys_post);
    if (d.user)
        write_lexicon(*d.user, us, lmap, rmap, left_lb, out.data() + h.off_usr_table, out.data() + h.off_usr_nodes,
                      out.data() + h.off_usr_post);
    uint32_t* uo = reinterpret_cast<uint32_t*>(out.data() + h.off_unk_off);
    for (uint32_t i = 0; i <= n_cat; ++i) uo[i] = uint32_t(d.unk.offsets[i]);
    uint32_t* ue = reinterpret_cast<uint32_t*>(out.data() + h.off_unk_ent);
    for (uint32_t i = 0; i < h.n_unk; ++i) {
        const UnkEntry& e = d.unk.entries[i];
        ue[2 * i] = uint32_t(lmap[e.left_id]) | (uint32_t(rmap[e.right_id]) << 16);
        ue[2 * i + 1] = pack_cost(e.word_cost, left_lb[e.left_id]);
    }
    for (int li = 0; li < 3; ++li) {
        uint32_t* fo = reinterpret_cast<uint32_t*>(out.data() + h.off_feat_off[li]);
        uint8_t* fb = out.data() + h.off_feat[li];
        uint16_t* pp = reinterpret_cast<uint16_t*>(out.data() + h.off_params[li]);
        if (li < 2) {
            const Lexicon* lx = lexs[li];
            if (!lx) {
                fo[0] = 0;
                continue;
            }
            for (uint32_t i = 0; i <= lx->num_words(); ++i) fo[i] = uint32_t(lx->feature_off[i] - lx->feature_off[0]);
            if (!lx->feature_blob.empty())
                std::memcpy(fb, lx->feature_blob.data() + lx->feature_off[0], lx->feature_off[lx->num_words()] - lx->feature_off[0]);
            for (uint32_t i = 0; i < lx->num_words(); ++i) {
                pp[4 * i] = lx->params[i].left_id;
                pp[4 * i + 1] = lx->params[i].right_id;
                pp[4 * i + 2] = uint16_t(lx->params[i].word_cost);
            }
        } else {
            uint32_t o = 0;
            for (uint32_t i = 0; i < d.unk.entries.size(); ++i) {
                const UnkEntry& e = d.unk.entries[i];
                fo[i] = o;
                if (!e.feature.empty()) std::memcpy(fb + o, e.feature.data(), e.feature.size());
                o += uint32_t(e.feature.size());
                pp[4 * i] = e.left_id;
                pp[4 * i + 1] = e.right_id;
                pp[4 * i + 2] = uint16_t(e.word_cost);
            }
            fo[d.unk.entries.size()] = o;
        }
    }
    {
        uint16_t* li = reinterpret_cast<uint16_t*>(out.data() + h.off_left_ids);
        uint16_t* ri = reinterpret_cast<uint16_t*>(out.data() + h.off_right_ids);
        for (uint32_t l = 0; l < nl; ++l) li[lmap[l]] = uint16_t(l);
        for (uint32_t r = 0; r < nr; ++r) ri[rmap[r]] = uint16_t(r);
    }
    if (raw) {  // feature rows move with the renumbered ids; the scorer is id-independent
        const size_t T = d.raw.feat_T;
        uint32_t* rf = reinterpret_cast<uint32_t*>(out.data() + h.off_right_feats);
        uint32_t* lf = reinterpret_cast<uint32_t*>(out.data() + h.off_left_feats);
        for (uint32_t r = 0; r < nr; ++r) std::memcpy(rf + size_t(rmap[r]) * T, d.raw.right_feats.data() + size_t(r) * T, T * 4);
        for (uint32_t l = 0; l < nl; ++l) std::memcpy(lf + size_t(lmap[l]) * T, d.raw.left_feats.data() + size_t(l) * T, T * 4);
        if (!d.raw.bases.empty()) std::memcpy(out.data() + h.off_bases, d.raw.bases.data(), d.raw.bases.size() * 4);
        if (!d.raw.checks.empty()) std::memcpy(out.data() + h.off_checks, d.raw.checks.data(), d.raw.checks.size() * 4);
        if (!d.raw.costs.empty()) std::memcpy(out.data() + h.off_costs, d.raw.costs.data(), d.raw.costs.size() * 4);
    }
    if (dual) {  // the reduced matrix keeps its own numbering; the per-id maps follow the renumbered ids
        std::memcpy(out.data() + h.off_matrix, d.matrix.data.data(), d.matrix.data.size() * 2);
        uint16_t* rc = reinterpret_cast<uint16_t*>(out.data() + h.off_right_conn);
        uint16_t* lc = reinterpret_cast<uint16_t*>(out.data() + h.off_left_conn);
        for (uint32_t r = 0; r < nr; ++r) rc[rmap[r]] = d.dual_right_map[r];
        for (uint32_t l = 0; l < nl; ++l) lc[lmap[l]] = d.dual_left_map[l];
    } else if (!raw) {
        // Stored transposed (mt[right][left]): K3's lanes share a predecessor's right id and differ in the left ids
        // of their candidates, so one request then reads one row.  Tiled so that the reads and the writes of a tile
        // stay within a few lines; the two permutations scatter one side of the copy whatever the order, so the
        // 240 M-entry unidic matrix is split over host threads (tiles of different left ids write different columns:
        // no two threads touch the same element)
        int16_t* dm = reinterpret_cast<int16_t*>(out.data() + h.off_matrix);
        const int16_t* sm = d.matrix.data.data();
        constexpr uint32_t TB = 64;
        const uint32_t n_tiles = (nl + TB - 1) / TB;
        auto work = [&](uint32_t t0, uint32_t t1) {
            for (uint32_t t = t0; t < t1; ++t) {
                const uint32_t l0 = t * TB, l1 = std::min(nl, l0 + TB);
                for (uint32_t r0 = 0; r0 < nr; r0 += TB) {
                    const uint32_t r1 = std::min(nr, r0 + TB);
                    for (uint32_t l = l0; l < l1; ++l) {
                        const int16_t* src = sm + size_t(l) * nr;
                        const size_t col = lmap[l];
                        for (uint32_t r = r0; r < r1; ++r) dm[size_t(rmap[r]) * nl + col] = src[r];
                    }
                }
            }
        };
        const uint32_t n_thr = size_t(nl) * nr < (1u << 22) ? 1u : std::min<uint32_t>(8, std::max<uint32_t>(1, std::thread::hardware_concurrency()));
        if (n_thr <= 1) {
            work(0, n_tiles);
        } else {
            std::vector<std::thread> th;
            for (uint32_t i = 0; i < n_thr; ++i)
                th.emplace_back(work, uint32_t(uint64_t(n_tiles) * i / n_thr), uint32_t(uint64_t(n_tiles) * (i + 1) / n_thr));
            for (auto& t : th) t.join();
        }
        reinterpret_cast<BlobHeader*>(out.data())->matrix_transposed = 1;
    }
}

}  // namespace vbt
