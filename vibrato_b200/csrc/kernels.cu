// Hand-written sm_100a kernels of the batched Viterbi tokenizer.
//
//   K1a count_chars     warp / sentence   UTF-8 validation + character count
//   K1b decode          warp / sentence   code points -> CharInfo, trie codes, c2b, groupable
//   K2  candidates      thread / char     common-prefix walks (user, system) + unknown words
//   K3  viterbi2        8 lanes / sentence left-to-right min-plus DP over the lattice + EOS
//       count_lattice   thread / sentence counted runs only: SURVEY.md §8(d) counters and connection-id counts,
//                                         read off the finished lattice
//   K4a backtrack_count thread / sentence length of the best path
//   K4b backtrack_write thread / sentence token records, in sentence order
//
// Everything is integer gather / compare work: no tensor cores.  Citations are relative to
// /root/reference/vibrato/src/ and name the reference routine whose RESULT each step reproduces.
#include "kernels.cuh"

#include <climits>

// A batch whose byte offsets k_count_chars refused is not touched by any later kernel: the sizes derived from
// the offsets (slots, workspace bounds) cannot be trusted.
#define VBT_STAND_DOWN_IF_REJECTED(b) \
    if (*(b).flags & kFlagsStandDown) return

namespace vbt {

namespace {

constexpr uint32_t kMask = 0x7FFFFFFFu;
constexpr uint32_t kFlag = 0x80000000u;
constexpr unsigned kFull = 0xFFFFFFFFu;

// CharInfo bit fields (dictionary/character.rs:10-24,72-94)
__device__ __forceinline__ uint32_t ci_cate(uint32_t ci) { return ci & 0x3FFFFu; }
__device__ __forceinline__ uint32_t ci_base(uint32_t ci) { return (ci >> 18) & 0xFFu; }
__device__ __forceinline__ bool ci_invoke(uint32_t ci) { return (ci >> 26) & 1u; }
__device__ __forceinline__ bool ci_group(uint32_t ci) { return (ci >> 27) & 1u; }
__device__ __forceinline__ uint32_t ci_length(uint32_t ci) { return ci >> 28; }

__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// K1a: characters per sentence + UTF-8 validity (what `&str` guarantees before worker.rs:34)
// ---------------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t utf8_len_checked(const uint8_t* p, unsigned long long i, unsigned long long len,
                                                     uint32_t c, bool& bad) {
    uint32_t L;
    if (c < 0x80) return 1;
    if (c >= 0xC2 && c <= 0xDF)
        L = 2;
    else if (c >= 0xE0 && c <= 0xEF)
        L = 3;
    else if (c >= 0xF0 && c <= 0xF4)
        L = 4;
    else {
        bad = true;
        return 1;
    }
    if (i + L > len) {
        bad = true;
        return 1;
    }
    uint32_t c1 = p[i + 1];
    if ((c1 & 0xC0) != 0x80) bad = true;
    if (L >= 3 && (p[i + 2] & 0xC0) != 0x80) bad = true;
    if (L == 4 && (p[i + 3] & 0xC0) != 0x80) bad = true;
    if (c == 0xE0 && c1 < 0xA0) bad = true;  // overlong
    if (c == 0xED && c1 > 0x9F) bad = true;  // surrogates
    if (c == 0xF0 && c1 < 0x90) bad = true;
    if (c == 0xF4 && c1 > 0x8F) bad = true;
    return L;
}

// Sentences per warp of the warp-per-sentence kernels (K1a, K1b, K4b): a warp walks a few consecutive sentences so
// that the grid has fewer, longer-lived blocks.
constexpr uint32_t kSentPerWarp = 4;

__device__ __forceinline__ void count_chars_one(const Batch& b, uint32_t s, uint32_t lane) {
    unsigned long long bo = b.byte_off[s], len = b.byte_off[s + 1] - bo;
    if (b.byte_off[s + 1] < bo || b.byte_off[s + 1] > b.total_bytes) {  // caller error: nothing of this sentence is read
        if (lane == 0) {
            atomicOr(b.flags, kFlagBadOffsets);
            b.n_slots[s] = 1;
        }
        return;
    }
    const uint8_t* p = b.utf8 + bo;
    unsigned long long nchar = 0, covered = 0;
    bool bad = false;
    for (unsigned long long i0 = 0; i0 < len; i0 += 32) {
        unsigned long long i = i0 + lane;
        if (i < len) {
            uint32_t c = p[i];
            if ((c & 0xC0) != 0x80) {
                covered += utf8_len_checked(p, i, len, c, bad);
                ++nchar;
            }
        }
    }
    nchar = warp_sum(nchar);
    covered = warp_sum(covered);
    bool any_bad = __any_sync(kFull, bad);
    if (lane == 0) {
        if (any_bad || covered != len || nchar >= 0xFFFFFFF0ull) {
            atomicOr(b.flags, kFlagUtf8Error);
            nchar = 0;  // keep the rest of the pipeline in bounds; the batch is rejected anyway
        }
        b.n_slots[s] = uint32_t(nchar) + 1;
        if (nchar > kPruneMaxChars) atomicOr(b.flags, kFlagLongSentence);
        if (b.counters) {
            atomicAdd(&b.counters[kCntU], len);
            atomicAdd(&b.counters[kCntC], nchar);
        }
    }
}

__global__ void __launch_bounds__(256) k_count_chars(Batch b) {
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
#pragma unroll 1
    for (uint32_t r = 0; r < kSentPerWarp; ++r) {
        const uint32_t s = w * kSentPerWarp + r;
        if (s >= b.n_sent) return;
        count_chars_one(b, s, lane);
    }
}

// ---------------------------------------------------------------------------------------------
// K1b: Sentence::compile (sentence.rs:34-71) for every sentence
// ---------------------------------------------------------------------------------------------

__device__ __forceinline__ void decode_one(const DictView& d, const Batch& b, uint32_t s, uint32_t lane) {
    unsigned long long bo = b.byte_off[s], len = b.byte_off[s + 1] - bo;
    const uint8_t* p = b.utf8 + bo;
    const uint32_t base = b.slot_off[s];
    const uint32_t n = b.slot_off[s + 1] - base - 1;
    if (n > 0) {  // n == 0 also covers a batch already flagged as invalid UTF-8
        uint32_t running = 0;
        for (unsigned long long i0 = 0; i0 < len; i0 += 32) {
            unsigned long long i = i0 + lane;
            uint32_t c = i < len ? p[i] : 0x80u;
            bool lead = (c & 0xC0) != 0x80;
            uint32_t m = __ballot_sync(kFull, lead);
            if (lead) {
                uint32_t idx = running + __popc(m & lanemask_lt());
                uint32_t c1 = i + 1 < len ? p[i + 1] : 0, c2 = i + 2 < len ? p[i + 2] : 0, c3 = i + 3 < len ? p[i + 3] : 0;
                uint32_t cp;  // compute_basic sentence.rs:40-46
                if (c < 0x80)
                    cp = c;
                else if (c < 0xE0)
                    cp = ((c & 0x1F) << 6) | (c1 & 0x3F);
                else if (c < 0xF0)
                    cp = ((c & 0x0F) << 12) | ((c1 & 0x3F) << 6) | (c2 & 0x3F);
                else
                    cp = ((c & 0x07) << 18) | ((c1 & 0x3F) << 12) | ((c2 & 0x3F) << 6) | (c3 & 0x3F);
                if (idx < n) {
                    uint32_t slot = base + idx;
                    b.byte_pos[slot] = uint32_t(i);
                    // CharProperty::char_info character.rs:112-116: out-of-table code points use entry 0
                    b.cinfo[slot] = __ldg(&d.chr2inf[cp < d.chr2inf_len ? cp : 0]);
                    b.code_sys[slot] = cp < d.sys_table_len ? __ldg(&d.sys_table[cp]) : kInvalidCode;
                    if (d.usr_table) b.code_usr[slot] = cp < d.usr_table_len ? __ldg(&d.usr_table[cp]) : kInvalidCode;
                    b.ends_cnt[slot] = idx == 0 ? 1u : 0u;  // BOS lives in ends[0] (lattice.rs:72-83)
                }
            }
            running += __popc(m);
        }
    }
    if (lane == 0) {  // sentinel slot == character position n
        uint32_t slot = base + n;
        b.byte_pos[slot] = uint32_t(len);
        b.cinfo[slot] = 0;
        b.groupable[slot] = 0;
        b.code_sys[slot] = kInvalidCode;
        if (d.usr_table) b.code_usr[slot] = kInvalidCode;
        b.ends_cnt[slot] = 0;
        b.info[slot] = make_uint2(0, 0);
    }
    __syncwarp();
    // compute_groupable sentence.rs:57-71: distance to the end of the run in which adjacent
    // characters share a category bit, solved per 32-character chunk from the right.
    uint32_t carry = 0;
    for (int k = int((n + 31) / 32) - 1; k >= 0; --k) {
        uint32_t c = uint32_t(k) * 32 + lane;
        bool valid = c < n;
        uint32_t ci = valid ? b.cinfo[base + c] : 0;
        uint32_t cn = (c + 1 < n) ? b.cinfo[base + c + 1] : 0;
        bool brk = valid && (c + 1 == n || (ci_cate(ci) & ci_cate(cn)) == 0);
        uint32_t bm = __ballot_sync(kFull, brk);
        uint32_t clen = min(32u, n - uint32_t(k) * 32);
        uint32_t m = bm >> lane;
        uint32_t g = m ? uint32_t(__ffs(m)) : (clen - lane) + carry;
        if (valid) b.groupable[base + c] = g;
        carry = __shfl_sync(kFull, g, 0);
    }
}

__global__ void __launch_bounds__(256) k_decode(DictView d, Batch b) {
    VBT_STAND_DOWN_IF_REJECTED(b);
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
#pragma unroll 1
    for (uint32_t r = 0; r < kSentPerWarp; ++r) {
        const uint32_t s = w * kSentPerWarp + r;
        if (s >= b.n_sent) return;
        decode_one(d, b, s, lane);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// K2: lattice candidates per start position = Tokenizer::add_lattice_edges (tokenizer.rs:141-199)
// ---------------------------------------------------------------------------------------------

struct WalkStats {
    uint32_t m, t, p, w, walks;
};

// Candidate sources of one start position — trie hits (a postings list each) and unknown-word spans (a run of
// unk.def entries each) — kept in shared memory between the counting walk and the fill, so that the dependent
// pointer chase through the double array is done once and the fill can deal the candidates of a whole warp to its
// lanes.  A segment = {kind | index, end slot} + its candidate count.  Column-major ([segment][thread]) keeps the
// accesses of a warp conflict-free.
constexpr uint32_t kMaxHits = 8;
constexpr uint32_t kSegUser = 0x80000000u, kSegUnk = 0x40000000u, kSegIndex = 0x3FFFFFFFu;
struct HitBuf {
    uint2* col;    // &hits[0][threadIdx.x]; stride blockDim.x
    uint8_t* cnt;  // &counts[0][threadIdx.x]; stride blockDim.x
    uint32_t stride;
    uint32_t n;  // segments seen; kMaxHits + 1 and beyond = does not fit (the fill then regenerates per thread)
    __device__ __forceinline__ void push(uint32_t v, uint32_t end, uint32_t count) {
        if (n < kMaxHits && count < 256u && (v & kSegIndex) == (v & ~(kSegUser | kSegUnk))) {
            col[n * stride] = make_uint2(v, end);
            cnt[n * stride] = uint8_t(count);
            ++n;
        } else {
            n = kMaxHits + 1;
        }
    }
};

// Lexicon::common_prefix_iterator (lexicon.rs:33-46): crawdad common-prefix search over the double
// array (trie.rs:49-56), then the postings of every hit (posting.rs:18-21) with their WordParams.
template <bool FILL, bool COUNT>
__device__ __forceinline__ uint32_t walk_lexicon(const uint4* __restrict__ nodes, uint32_t num_nodes,
                                                 const uint4* __restrict__ post,
                                                 const uint32_t* __restrict__ codes,
                                                 const uint32_t* __restrict__ groupable, uint32_t sw, uint4* out,
                                                 uint32_t* ends_cnt, WalkStats& st, HitBuf* hb = nullptr,
                                                 uint32_t lex_flag = 0) {
    if (num_nodes == 0) return 0;
    uint32_t count = 0, node = 0, d = 0, hits = 0;
    uint32_t nbase = __ldg(&nodes[0].x);
    uint32_t q = sw;
    for (;; ++q) {
        uint32_t code = codes[q];
        if (code == kInvalidCode) break;  // unmapped character or the sentence's sentinel
        if (nbase & kFlag) break;         // a leaf has no children
        uint32_t child = nbase ^ code;
        if (child >= num_nodes) break;
        const uint4 nd = __ldg(&nodes[child]);  // one 16-byte load per step: base, check, and the key ending here
        if ((nd.y & kMask) != node) break;
        node = child;
        nbase = nd.x;
        ++d;
        if (nd.z == kNone) continue;
        const uint32_t v = nd.z;
        const uint32_t plen = nd.w;
        if (!FILL && hb) hb->push(v | lex_flag, q + 1, plen);
        if (FILL) {
            for (uint32_t j = 0; j < plen; ++j) {
                uint4 e = __ldg(&post[v + 1 + j]);
                e.w = q + 1;
                out[count + j] = e;
            }
            atomicAdd(&ends_cnt[q + 1], plen);
        }
        count += plen;
        ++hits;
        if (COUNT) {
            st.p += 1 + plen;
            st.w += plen;
        }
    }
    if (COUNT) {
        uint32_t f = groupable[q] != 0 ? 1u : 0u;  // 0 when the walk ran off the end of the sentence
        st.m += d + f;
        st.t += d + f + hits;
        st.walks += 1;
    }
    return count;
}

// UnkHandler::gen_unk_words (unknown.rs:69-116) with scan_entries (:119-137).
template <bool FILL>
__device__ __forceinline__ uint32_t gen_unknown(const DictView& d, uint32_t sw, uint32_t ci, uint32_t g,
                                                bool has_matched, uint4* out, uint32_t* ends_cnt, HitBuf* hb = nullptr) {
    if (has_matched && !ci_invoke(ci)) return 0;
    const uint32_t e0 = __ldg(&d.unk_off[ci_base(ci)]), e1 = __ldg(&d.unk_off[ci_base(ci) + 1]);
    const uint32_t ne = e1 - e0;
    uint32_t count = 0;
    auto span = [&](uint32_t end) {
        if (FILL) {
            for (uint32_t j = 0; j < ne; ++j) {
                uint2 e = __ldg(&d.unk_ent[e0 + j]);
                // unknown.rs:133 `word_id as u16`, LexType::Unknown
                out[count + j] = make_uint4(e.x, e.y, (2u << 30) | ((e0 + j) & 0xFFFFu), end);
            }
            if (ne) atomicAdd(&ends_cnt[end], ne);
        }
        if (!FILL && hb && ne) hb->push(kSegUnk | e0, end, ne);
        count += ne;
    };
    bool grouped = false;
    if (ci_group(ci)) {
        grouped = true;
        if ((unsigned long long)(g - 1) <= d.max_grouping) {  // :91-93
            span(sw + g);
            has_matched = true;
        }
    }
    uint32_t lim = min(ci_length(ci), g);
    for (uint32_t i = 1; i <= lim; ++i) {
        if (grouped && i == g) continue;
        span(sw + i);  // sw + i <= sentence length because i <= groupable
        has_matched = true;
    }
    if (!has_matched) span(sw + 1);  // :112-115
    return count;
}

__global__ void __launch_bounds__(256) k_candidates(DictView d, Batch b) {
    constexpr bool COUNT = false;  // M/T/P/W are produced by k_count_lattice in counted runs
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31;
    // A rejected batch (see VBT_STAND_DOWN_IF_REJECTED) leaves every thread out of range.  The flag word is read
    // next to the slot total instead of in front of it: with 256-thread blocks that live for one trie walk, a
    // dependent extra round trip at the top costs 8 % of this kernel (profiles/r01e_k3_variants_ab.md).
    const uint32_t batch_flags = *b.flags;
    const uint32_t total_slots = b.slot_off[b.n_sent];
    if (slot == 0 && total_slots > b.launch_slots) atomicOr(b.flags, kFlagSlotsOverflow);
    const bool in_range = slot < total_slots && !(batch_flags & kFlagBadOffsets);
    uint32_t g0 = in_range ? b.groupable[slot] : 0;
    bool active = in_range && g0 != 0;
    uint32_t sw = slot, skip = 0, flags = 0, ci = 0, g = 0;
    WalkStats st{0, 0, 0, 0, 0};
    if (active) {
        uint32_t ci0 = b.cinfo[slot];
        if (ci_cate(ci0) & d.space_mask) {  // tokenizer.rs:117-125: skip the groupable run at a space
            skip = g0;
            sw = slot + skip;
        }
        g = skip ? b.groupable[sw] : g0;
        if (g == 0) {  // start_word == len: tokenizer.rs:128-130
            flags = kInfoTrailing;
            active = false;
        } else {
            ci = skip ? b.cinfo[sw] : ci0;
        }
    }
    uint32_t cnt = 0;
    bool matched = false;
    __shared__ uint2 s_hits[kMaxHits][256];
    __shared__ uint8_t s_seg_cnt[kMaxHits][256];
    HitBuf hb{&s_hits[0][threadIdx.x], &s_seg_cnt[0][threadIdx.x], 256, 0};
    if (active) {
        uint32_t cu = 0;
        if (d.usr_table)
            cu = walk_lexicon<false, COUNT>(d.usr_nodes, d.usr_num_nodes, d.usr_post, b.code_usr, b.groupable, sw,
                                            nullptr, nullptr, st, &hb, kSegUser);
        uint32_t cs = walk_lexicon<false, COUNT>(d.sys_nodes, d.sys_num_nodes, d.sys_post, b.code_sys, b.groupable,
                                                 sw, nullptr, nullptr, st, &hb, 0);
        matched = (cu + cs) != 0;
        uint32_t ck = gen_unknown<false>(d, sw, ci, g, matched, nullptr, nullptr, &hb);
        if (COUNT) st.w += ck;
        cnt = cu + cs + ck;
    }
    // Block-aggregated allocation from the candidate pool: a scan inside each warp, the eight warp totals through
    // shared memory, ONE atomicAdd per block.  (One atomic per warp was 1.3 M same-address atomics per batch, and
    // every warp sat on the round trip of its own; the pool also comes out in slot order block by block.)
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t v = __shfl_up_sync(kFull, incl, o);
        if (lane >= uint32_t(o)) incl += v;
    }
    __shared__ uint32_t s_warp_total[8];
    __shared__ unsigned long long s_block_base;
    const uint32_t wid = threadIdx.x >> 5;
    if (lane == 31) s_warp_total[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int i = 0; i < 8; ++i) {  // warp totals -> exclusive offsets inside the block
            const uint32_t t = s_warp_total[i];
            s_warp_total[i] = run;
            run += t;
        }
        s_block_base = run ? atomicAdd(b.pool_ctr, (unsigned long long)run) : 0ull;
        if (s_block_base + run > (unsigned long long)b.cand_cap) atomicOr(b.flags, kFlagPoolOverflow);
    }
    __syncthreads();
    const unsigned long long wbase = s_block_base + s_warp_total[wid];
    const uint32_t warp_total = __shfl_sync(kFull, incl, 31);
    const bool fits = wbase + warp_total <= (unsigned long long)b.cand_cap;
    uint32_t ptr = uint32_t(wbase) + (incl - cnt);
    if (in_range && g0 != 0) {
        const bool special = (skip | flags) != 0;
        b.info[slot] = make_uint2(ptr, (fits ? cnt : 0) | (special ? kInfoSpecial : 0u));
        if (special) b.info_ex[slot] = make_uint2(skip, flags);
    }
    // Fill.  Usual case: every position of the warp kept its sources in the segment buffer; the warp's candidates
    // (contiguous in the pool, in position order) are then dealt to the 32 lanes as ONE list — lane i writes entries
    // i, i + 32, ...: full-width, coalesced stores and loads that walk postings lists side by side, instead of
    // every lane copying its own run of ~7 candidates with the others idle.  An entry finds its position by a
    // binary search over the warp's inclusive counts (shuffles) and its segment by a short scan of that position's
    // segment counts.
    const bool pooled = !__any_sync(kFull, hb.n > kMaxHits);
    if (pooled) {
        if (fits) {
            if (active)
                for (uint32_t h = 0; h < hb.n; ++h) atomicAdd(&b.ends_cnt[hb.col[h * hb.stride].y], uint32_t(hb.cnt[h * hb.stride]));
            const uint32_t col0 = threadIdx.x & ~31u;
            for (uint32_t e0 = 0; e0 < warp_total; e0 += 32) {
                const uint32_t e = e0 + lane;
                uint32_t t = 0;  // owner = number of positions whose inclusive count is <= e
#pragma unroll
                for (uint32_t step = 16; step; step >>= 1) {
                    const uint32_t v = __shfl_sync(kFull, incl, t + step - 1);
                    if (v <= e) t += step;
                }
                t = min(t, 31u);
                uint32_t local = e - __shfl_sync(kFull, incl - cnt, t);
                if (e < warp_total) {
                    uint32_t h = 0;
                    uint32_t c = s_seg_cnt[0][col0 + t];
                    while (local >= c) {  // e < warp_total: the owner has a segment that holds it
                        local -= c;
                        ++h;
                        c = s_seg_cnt[h][col0 + t];
                    }
                    const uint2 seg = s_hits[h][col0 + t];
                    uint4 rec;
                    if (seg.x & kSegUnk) {  // unknown.rs:133 `word_id as u16`, LexType::Unknown
                        const uint32_t id = (seg.x & kSegIndex) + local;
                        const uint2 ue = __ldg(&d.unk_ent[id]);
                        rec = make_uint4(ue.x, ue.y, (2u << 30) | (id & 0xFFFFu), seg.y);
                    } else {
                        const uint4* __restrict__ post = (seg.x & kSegUser) ? d.usr_post : d.sys_post;
                        rec = __ldg(&post[(seg.x & kSegIndex) + 1 + local]);  // the candidate record, end slot still open
                        rec.w = seg.y;
                    }
                    b.cand[uint32_t(wbase) + e] = rec;
                }
            }
        }
    } else if (active && fits && cnt) {  // some position has more sources than the buffer holds: regenerate per thread
        uint4* out = b.cand + ptr;
        uint32_t w = 0;
        if (d.usr_table)
            w += walk_lexicon<true, false>(d.usr_nodes, d.usr_num_nodes, d.usr_post, b.code_usr, b.groupable, sw,
                                           out + w, b.ends_cnt, st);
        w += walk_lexicon<true, false>(d.sys_nodes, d.sys_num_nodes, d.sys_post, b.code_sys, b.groupable, sw,
                                       out + w, b.ends_cnt, st);
        gen_unknown<true>(d, sw, ci, g, matched, out + w, b.ends_cnt);
    }
    (void)st;
}

// ---------------------------------------------------------------------------------------------
// K3: Tokenizer::build_lattice_inner (tokenizer.rs:94-139) + Lattice::insert_node / search_min_node /
//     insert_eos (lattice.rs:85-151).
//
// 8 lanes per sentence (4 sentences per warp, walking their start positions in lockstep, one position after
// the other), built around what the r01f profile showed to be the limits — warp-instruction issue and the LSU data
// pipe of the L1 (shuffles, spills and gathers all queue there):
//   * per position the candidates of the warp's sentences are dealt to the 32 lanes as one pool, lane = candidate;
//     the typical position has ~7 candidates and ~8 predecessors;
//   * the predecessors {cost, right} of a position are staged once in shared memory and read back two at a time
//     with one LDS.128 (a broadcast inside the group) instead of two SHFL per predecessor;
//   * the gather address is one multiply-add on a per-candidate column pointer (the matrix is stored transposed);
//   * no state is carried across positions except three slot numbers: nothing spills at 32 registers;
//   * exact lower-bound pruning (PRUNE): every candidate record carries lb = min over ALL right ids of
//     M[right][left], so a predecessor with cost + lb > best-so-far cannot reach the minimum, not even tie it,
//     and its gather is skipped.  Predecessors are still visited in row order with `<=`, so the LAST minimal one
//     wins exactly as in Lattice::search_min_node (lattice.rs:129-151).  The bound arithmetic assumes that no i32
//     addition wraps: batches holding a sentence longer than kPruneMaxChars characters take the unpruned path,
//     which keeps the reference's wrapping adds.
// ---------------------------------------------------------------------------------------------

// ConnectorCost::cost(right_id, left_id) for one fixed left id (one candidate).
template <int CONN>
struct ConnRow;

template <>
struct ConnRow<0> {  // MatrixConnector::cost (matrix_connector.rs:79-85,121-124): one 2-byte gather
    // The image stores the matrix transposed, mt[right][left]: the lanes of a group share the predecessor's
    // right id and differ in their candidates' left ids, so with usage-sorted ids the frequent candidates of
    // one request fall into the same 128-byte line of row `right` instead of one line per candidate row.
    uint32_t off;  // the image builder refuses matrices of 2^32 entries or more, so 32-bit indices suffice
    __device__ __forceinline__ ConnRow(const DictView& d, uint32_t left) : off(left * d.conn_stride_left) {}
    __device__ __forceinline__ int32_t cost(const DictView& d, uint32_t right) const {
        return int32_t(__ldg(d.matrix + (off + right * d.conn_stride_right)));
    }
};

template <>
struct ConnRow<1> {  // RawConnector::cost (raw_connector.rs:155-160) = Scorer::accumulate_cost (scorer.rs:240-267)
    const uint32_t* __restrict__ lf;
    __device__ __forceinline__ ConnRow(const DictView& d, uint32_t left) : lf(d.left_feats + size_t(left) * d.feat_T) {}
    __device__ __forceinline__ int32_t cost(const DictView& d, uint32_t right) const {
        const uint32_t* __restrict__ rf = d.right_feats + size_t(right) * d.feat_T;
        uint32_t score = 0;
        for (uint32_t t = 0; t < d.feat_T; ++t) {
            const uint32_t key1 = __ldg(rf + t), key2 = __ldg(lf + t);
            if (key1 < d.n_bases) {  // INVALID_FEATURE_ID (0x7fffffff) never passes
                const uint32_t pos = __ldg(d.sc_bases + key1) ^ key2;
                if (pos < d.n_checks && __ldg(d.sc_checks + pos) == key1) score += uint32_t(__ldg(d.sc_costs + pos));
            }
        }
        return int32_t(score);
    }
};

template <>
struct ConnRow<2> {  // DualConnector::cost (dual_connector.rs:269-280): reduced-matrix gather + one 8-lane scorer row
    const int16_t* __restrict__ row;
    uint4 l0, l1;  // the candidate's eight raw feature ids stay in registers across its predecessors
    __device__ __forceinline__ ConnRow(const DictView& d, uint32_t left)
        : row(d.matrix + size_t(__ldg(d.left_conn + left)) * d.num_right) {
        const uint4* __restrict__ lf = reinterpret_cast<const uint4*>(d.left_feats + size_t(left) * 8);
        l0 = __ldg(lf);
        l1 = __ldg(lf + 1);
    }
    __device__ __forceinline__ uint32_t lane(const DictView& d, uint32_t key1, uint32_t key2) const {
        if (key1 < d.n_bases) {
            const uint32_t pos = __ldg(d.sc_bases + key1) ^ key2;
            if (pos < d.n_checks && __ldg(d.sc_checks + pos) == key1) return uint32_t(__ldg(d.sc_costs + pos));
        }
        return 0;
    }
    __device__ __forceinline__ int32_t cost(const DictView& d, uint32_t right) const {
        const uint4* __restrict__ rf = reinterpret_cast<const uint4*>(d.right_feats + size_t(right) * 8);
        const uint4 r0 = __ldg(rf), r1 = __ldg(rf + 1);
        uint32_t score = uint32_t(int32_t(__ldg(row + __ldg(d.right_conn + right))));
        score += lane(d, r0.x, l0.x) + lane(d, r0.y, l0.y) + lane(d, r0.z, l0.z) + lane(d, r0.w, l0.w);
        score += lane(d, r1.x, l1.x) + lane(d, r1.y, l1.y) + lane(d, r1.z, l1.z) + lane(d, r1.w, l1.w);
        return int32_t(score);
    }
};

// k_viterbi2's shape.  Other block sizes and prefetch distances measured no different (profiles/r02_k3_variants_ab.md).
constexpr int kV2Lanes = 8;                        // lanes of a warp per sentence
constexpr uint32_t kV2SentPerWarp = 32 / kV2Lanes;
constexpr int kV2Warps = 4;                        // warps per block
constexpr int kV2MinBlocks = 64 / kV2Warps;        // 64 warps per SM = 32 registers per thread
constexpr uint32_t kV2PrefetchDist = 8;            // candidate records ahead of the current position

constexpr int kPredCap = 32;                             // predecessors staged per pass
constexpr int32_t kPredSentinel = INT32_MAX - 70000;     // + any i16 stays below INT32_MAX and above every real best

// Connection cost into one fixed left id for k_viterbi2.
template <int CONN>
struct ConnCol;
template <>
struct ConnCol<0> {
    // The engine places the matrix so that it does not cross a 4 GiB boundary (DictView::matrix_window): the
    // high address word is then the same for every entry and a lookup is ONE multiply-add on the low word,
    //     lo = right * (2 * stride_right) + colbase,   colbase = lo(matrix) + 2 * stride_left * left,
    // followed by the 2-byte load.  colbase / stride / hi are opaque (volatile asm) so that the compiler keeps
    // them in registers across the predecessor loop instead of recomputing them from the left id per lookup,
    // which is what it does when squeezed into 32 registers.
    uint32_t colbase, stride2, hi, zero;
    __device__ __forceinline__ ConnCol(const DictView& d, uint32_t left) {
        zero = d.opaque_zero;
        const unsigned long long base = reinterpret_cast<unsigned long long>(d.matrix);
        asm volatile("mad.lo.u32 %0, %1, %2, %3;" : "=r"(colbase) : "r"(left), "r"(d.conn_stride_left * 2u), "r"(uint32_t(base)));
        stride2 = d.conn_stride_right * 2u;  // uniform: the compiler may keep these two in uniform registers
        hi = uint32_t(base >> 32);
    }
    __device__ __forceinline__ int32_t cost(const DictView&, uint32_t right) const {
        int32_t m;
        asm("{\n\t.reg .u32 lo;\n\t.reg .u64 a;\n\tmad.lo.u32 lo, %1, %2, %3;\n\tmov.b64 a, {lo, %4};\n\t"
            "ld.global.nc.s16 %0, [a];\n\t}"
            : "=r"(m)
            : "r"(right), "r"(stride2), "r"(colbase), "r"(hi));
        return m;
    }
    // Two predecessors of Lattice::search_min_node, staged at shared address `pp` as {cost, right} pairs.  Phase 1
    // tests every one of them (PRUNE: cost + lb <= best, lb = cost_word >> 16; otherwise: its address lies below
    // `plim`, the end of this lane's row) and issues the surviving 2-byte gathers together; phase 2 folds them in
    // row order with `<=`, so the LAST minimum wins.  A bound that is one batch old is still a bound: `best` only
    // falls.  The shared address of the winner is its token (`besttok`).
#define VBT_V2_DECL(i) ".reg .pred p" #i ";\n\t.reg .s32 c" #i ", m" #i ";\n\t.reg .u32 r" #i ", l" #i ";\n\t.reg .u64 a" #i ";\n\t"
#define VBT_V2_TEST_PRUNE(i) "add.s32 t, c" #i ", lb;\n\tsetp.le.s32 p" #i ", t, %0;\n\t"
#define VBT_V2_TEST_PLAIN(i) "add.u32 l" #i ", %2, " #i "*8;\n\tsetp.lt.u32 p" #i ", l" #i ", %3;\n\t"
#define VBT_V2_LOAD(i) \
    "mad.lo.u32 l" #i ", r" #i ", %4, %5;\n\tmov.b64 a" #i ", {l" #i ", %6};\n\t@p" #i " ld.global.nc.s16 m" #i ", [a" #i "];\n\t"
#define VBT_V2_FOLD(i) \
    "@p" #i " add.s32 t, c" #i ", m" #i ";\n\tsetp.le.and.s32 q, t, %0, p" #i ";\n\tselp.s32 %0, t, %0, q;\n\t" \
    "add.u32 k, %2, " #i "*8;\n\tselp.u32 %1, k, %1, q;\n\t"
#define VBT_V2_HEAD "{\n\t.reg .pred q;\n\t.reg .s32 t, lb;\n\t.reg .u32 k;\n\t"
#define VBT_V2_OPERANDS \
    : "+r"(best), "+r"(besttok) : "r"(pp), "r"(PRUNE ? cost_word : plim), "r"(stride2), "r"(colbase), "r"(hi)
    // `zero` is a run-time zero the compiler cannot see through: the first fold reads m0 | (m1 & zero) = m0, one
    // LOP3 that needs BOTH gathers, so the two loads are issued back to back (left alone, ptxas at 32 registers
    // sinks the second load below the first fold and the two round trips serialise).
#define VBT_V2_FOLD0_JOIN(j) \
    "lop3.b32 k, m0, m" #j ", %7, 0xF8;\n\t@p0 add.s32 t, c0, k;\n\tsetp.le.and.s32 q, t, %0, p0;\n\t" \
    "selp.s32 %0, t, %0, q;\n\tselp.u32 %1, %2, %1, q;\n\t"
    template <bool PRUNE>
    __device__ __forceinline__ void batch2(uint32_t pp, uint32_t cost_word, uint32_t plim, int32_t& best,
                                           uint32_t& besttok) const {
        if (PRUNE)
            asm volatile(VBT_V2_HEAD VBT_V2_DECL(0) VBT_V2_DECL(1) "ld.shared.v4.b32 {c0, r0, c1, r1}, [%2];\n\tshr.s32 lb, %3, 16;\n\t"
                         VBT_V2_TEST_PRUNE(0) VBT_V2_TEST_PRUNE(1) VBT_V2_LOAD(0) VBT_V2_LOAD(1)  //
                         VBT_V2_FOLD0_JOIN(1) VBT_V2_FOLD(1) "}" VBT_V2_OPERANDS, "r"(zero));
        else
            asm volatile(VBT_V2_HEAD VBT_V2_DECL(0) VBT_V2_DECL(1) "ld.shared.v4.b32 {c0, r0, c1, r1}, [%2];\n\t"
                         VBT_V2_TEST_PLAIN(0) VBT_V2_TEST_PLAIN(1) VBT_V2_LOAD(0) VBT_V2_LOAD(1)  //
                         VBT_V2_FOLD0_JOIN(1) VBT_V2_FOLD(1) "}" VBT_V2_OPERANDS, "r"(zero));
    }
};

// Raw / Dual connectors, and the matrix with 64-bit addresses (CONN 3: a matrix that crosses a 4 GiB address
// boundary, and the `viterbi_kernel = 0` check of that path): plain C++ over ConnRow::cost, same interface.
template <int CONN>
struct ConnCol : ConnRow<CONN == 3 ? 0 : CONN> {
    using Row = ConnRow<CONN == 3 ? 0 : CONN>;
    const DictView& dv;
    __device__ __forceinline__ ConnCol(const DictView& d, uint32_t left) : Row(d, left), dv(d) {}
    template <bool PRUNE>
    __device__ __forceinline__ void batch1(uint32_t pp, uint32_t, uint32_t plim, int32_t& best, uint32_t& besttok) const {
        if (pp < plim) {
            int2 pr;
            asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(pr.x), "=r"(pr.y) : "r"(pp));
            const int32_t v = int32_t(uint32_t(pr.x) + uint32_t(this->cost(dv, uint32_t(pr.y))));  // i32 wrapping add
            if (v <= best) {
                best = v;
                besttok = pp;
            }
        }
    }
    template <bool PRUNE>
    __device__ __forceinline__ void batch2(uint32_t pp, uint32_t cw, uint32_t plim, int32_t& best, uint32_t& besttok) const {
#pragma unroll
        for (int i = 0; i < 2; ++i) batch1<PRUNE>(pp + 8 * i, cw, plim, best, besttok);
    }
};

// Shared-memory window of one warp of k_viterbi2: a staging row per sentence ({cost, right} of the predecessors, up
// to kPredCap per pass plus padding to whole batches; the odd multiple of 32 bytes skews the rows across the banks),
// and per sentence the descriptor of its current position {cand_ptr, slot, row offset, K} and its candidate count.
struct V2Shared {
    static constexpr uint32_t kRowBytes = (kPredCap + 4) * 8;
    int2 rows[kV2SentPerWarp][kPredCap + 4];
    uint4 desc[kV2SentPerWarp];
    uint32_t cnt[8];
};

template <int CONN, bool PRUNE, bool SPACE>
__device__ __forceinline__ void viterbi2_sweep(const DictView& d, const Batch& b, const uint32_t sw /* shared-window address of this warp's V2Shared */) {
    constexpr uint32_t kRowBytes = V2Shared::kRowBytes;
    constexpr uint32_t kDescOff = kV2SentPerWarp * kRowBytes, kCntOff = kDescOff + kV2SentPerWarp * 16;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gl = lane % kV2Lanes, sub = lane / kV2Lanes;
    const uint32_t s = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * kV2SentPerWarp + sub;

    uint32_t slot = 0, slot_end = 0;
    if (s < b.n_sent) {
        slot = b.slot_off[s];
        slot_end = b.slot_off[s + 1] - 1;
        if (gl == 0) {
            if (slot == slot_end) {  // Worker::tokenize returns early on an empty sentence (worker.rs:50-52)
                b.eos[s] = make_uint4(kNone, 0, 0, 0);
            } else {  // Lattice::insert_bos (lattice.rs:72-83): right_id 0, cost 0
                const uint32_t eo = b.ends_meta[slot].x;
                b.ends_hot[eo] = make_int2(0, 0);
                b.ends_cold[eo] = make_uint4(kNone, kNone, kNone, 0);
                b.ends_meta[slot].y = eo + 1;
            }
        }
    }
    __syncwarp();

    uint32_t skip_slot = slot;
    while (__any_sync(kFull, slot < slot_end)) {
        uint32_t K = 0, eo = 0, cptr = 0, ncand = 0;
        if (slot < slot_end) {  // two independent loads, one round trip
            const uint2 m = b.ends_meta[slot];
            const uint2 inf = b.info[slot];
            eo = m.x;
            K = m.y - m.x;
            // positions inside a skipped space run are never start_node; K == 0: has_previous_node fails
            if ((!SPACE || slot >= skip_slot) && K != 0) {  // (lattice.rs:155-157, tokenizer.rs:110-114)
                cptr = inf.x;
                ncand = inf.y;
            }
        }
        if (SPACE && (ncand & kInfoSpecial)) {
            ncand &= ~kInfoSpecial;
            const uint2 ex = b.info_ex[slot];
            if (ex.y & kInfoTrailing) {  // tokenizer.rs:128-130: EOS starts here, the sweep ends
                slot_end = slot;
                ncand = 0;
            } else if (ex.x) {
                skip_slot = slot + ex.x + 1;  // next start_node = start_word + 1 (tokenizer.rs:134-135)
            }
        }
        if (ncand == 0) K = 0;
        const uint32_t max_k = __reduce_max_sync(kFull, K);
        // K2 hands out the candidate pool in position order: pull the line of the positions ahead towards L1
        if (ncand && gl == 0 && cptr + ncand + kV2PrefetchDist < b.cand_cap)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(b.cand + cptr + ncand + kV2PrefetchDist));
        // The candidates of the warp's sentences are dealt to the 32 lanes as ONE pool (sentence after sentence):
        // a position with 3 candidates next to one with 13 fills half a warp, not two rounds of 8-lane groups.
        // Every group publishes its position; a lane then finds which sentence its pool index falls into.
        if (gl == 0) {
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sw + kDescOff + sub * 16u), "r"(cptr), "r"(slot),
                         "r"(eo), "r"(K)
                         : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(sw + kCntOff + sub * 4u), "r"(ncand) : "memory");
        }
        const uint32_t total = __reduce_add_sync(kFull, gl == 0 ? ncand : 0u);
        // Staging of the predecessors {cost, right} of every sentence's row, padded with sentinels to whole batches.
        // In the usual case (no row longer than kPredCap) it is started here with asynchronous copies (cp.async:
        // global -> shared without a register or a scoreboard entry in between) so that it overlaps the loads of
        // the candidates below; the copies are awaited right before the first batch.  Rows are 8-byte aligned only,
        // which rules out the 16-byte granular bulk copies (cp.async.bulk).
        const bool one_pass = max_k <= uint32_t(kPredCap);
        if (one_pass && total) {
            const uint32_t n_stage = (max_k + 1u) & ~1u;
            const uint32_t own = sw + sub * kRowBytes;
#pragma unroll 1
            for (uint32_t k = gl; k < n_stage; k += kV2Lanes) {
                if (k < K)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(own + k * 8u), "l"(b.ends_hot + eo + k) : "memory");
                else
                    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(own + k * 8u), "r"(kPredSentinel), "r"(0) : "memory");
            }
        }
        __syncwarp();
        for (uint32_t q0 = 0; q0 < total; q0 += 32) {
            const uint32_t q = q0 + lane;
            const bool valid = q < total;
            uint32_t s2 = 0, before = 0;
            {
                bool adv = true;
#pragma unroll
                for (uint32_t i = 0; i + 1 < kV2SentPerWarp; ++i) {
                    uint32_t c;
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(c) : "r"(sw + kCntOff + i * 4u));
                    adv = adv && q >= before + c;
                    if (adv) {
                        before += c;
                        s2 = i + 1;
                    }
                }
            }
            uint4 ds;  // {cand_ptr, slot, row offset, K} of the sentence this lane's candidate belongs to
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(ds.x), "=r"(ds.y), "=r"(ds.z), "=r"(ds.w)
                         : "r"(sw + kDescOff + s2 * 16u));
            uint4 cd = make_uint4(0, 0, 0, 0);
            uint32_t nxt = 0;
            if (valid) {
                cd = b.cand[ds.x + (q - before)];
                nxt = b.ends_meta[cd.w].y;  // next free entry of the row the node ends in: independent of the search
            }
            const ConnCol<CONN> conn(d, cd.x & 0xFFFFu);
            // Lattice::search_min_node (lattice.rs:129-151): `<=` keeps the LAST minimum
            int32_t best = (PRUNE && !valid) ? INT32_MIN : INT32_MAX;  // INT32_MIN: nothing passes the bound
            uint32_t bestk = 0;
#pragma unroll 1
            for (uint32_t k0 = 0; k0 < max_k; k0 += kPredCap) {
                // This pass covers predecessors [k0, k0 + kc) of every row, staged by the row's own group and padded
                // with sentinels to whole batches.
                const uint32_t kc = min(uint32_t(kPredCap), max_k - k0);
                const uint32_t n_stage = (kc + 1u) & ~1u;
                if (one_pass) {
                    if (q0 == 0) {  // the copies started above have had the candidates' round trip to arrive
                        asm volatile("cp.async.wait_all;" ::: "memory");
                        __syncwarp();
                    }
                } else {  // rows longer than kPredCap: pass after pass, staged synchronously
                    __syncwarp();
                    const uint32_t own = sw + sub * kRowBytes;
#pragma unroll 1
                    for (uint32_t k = gl; k < n_stage; k += kV2Lanes) {
                        int2 pr = make_int2(kPredSentinel, 0);
                        if (k0 + k < K) pr = b.ends_hot[eo + k0 + k];
                        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(own + k * 8u), "r"(pr.x), "r"(pr.y) : "memory");
                    }
                    __syncwarp();
                }
                // the shared address of a predecessor doubles as its token: index = k0 + (token - row) / 8
                const uint32_t row = sw + s2 * kRowBytes;
                const uint32_t plim = row + (valid ? min(ds.w - min(ds.w, k0), kc) : 0u) * 8u;  // end of this lane's row
                uint32_t besttok = kNone;
                const uint32_t pend = row + n_stage * 8u;
#pragma unroll 1
                for (uint32_t pp = row; pp < pend; pp += 16u) conn.template batch2<PRUNE>(pp, cd.y, plim, best, besttok);
                if (besttok != kNone) bestk = k0 + ((besttok - row) >> 3);
            }
            // Lattice::insert_node (lattice.rs:103-127): push into ends[end_word] in candidate order.
            // End slots of different sentences never coincide, so one warp-wide match suffices.
            const uint32_t vmask = __ballot_sync(kFull, valid);
            if (valid) {
                const uint32_t peers = __match_any_sync(vmask, cd.w);
                const uint32_t idx = nxt + __popc(peers & lanemask_lt());
                const int32_t cost = int32_t(uint32_t(best) + uint32_t(int32_t(int16_t(cd.y & 0xFFFFu))));
                b.ends_hot[idx] = make_int2(cost, int32_t(cd.x >> 16));
                // lattice.rs:144 keeps the predecessor index as u16
                b.ends_cold[idx] = make_uint4(ds.y, ds.z + (bestk & 0xFFFFu), cd.z, uint32_t(cost));
                if (idx == nxt) b.ends_meta[cd.w].y = nxt + __popc(peers);
            }
            __syncwarp();
        }
        if (slot < slot_end) ++slot;
    }

    // Lattice::insert_eos (lattice.rs:85-101): left_id 0, no word cost; lanes of the group = predecessors
    {
        const bool has_sentence = s < b.n_sent;
        const uint32_t base = has_sentence ? b.slot_off[s] : 0;
        const uint32_t n = has_sentence ? b.slot_off[s + 1] - 1 - base : 0;
        const uint32_t eos_start = slot_end - base;  // n, or the start of the trailing space run
        uint32_t K = 0, eo = 0;
        if (n > 0) {
            const uint2 m = b.ends_meta[slot_end];
            eo = m.x;
            K = m.y - m.x;
        }
        // minimise the signed 64-bit key (cost << 32 | ~index): smallest cost, then the LARGEST index
        // among ties — the `<=` rule of search_min_node
        long long bestkey = LLONG_MAX;
        const ConnCol<CONN> conn_eos(d, 0);  // BOS_EOS_CONNECTION_ID (common.rs:18)
        const uint32_t max_k = __reduce_max_sync(kFull, K);
        for (uint32_t k0 = 0; k0 < max_k; k0 += kV2Lanes) {
            long long key = LLONG_MAX;
            if (k0 + gl < K) {
                int2 pr = b.ends_hot[eo + k0 + gl];
                int32_t v = int32_t(uint32_t(pr.x) + uint32_t(conn_eos.cost(d, uint32_t(pr.y))));
                key = (long long)(((unsigned long long)uint32_t(v) << 32) | (unsigned long long)(~(k0 + gl)));
            }
#pragma unroll
            for (int o = kV2Lanes / 2; o > 0; o >>= 1) key = min(key, __shfl_xor_sync(kFull, key, o, kV2Lanes));
            bestkey = min(bestkey, key);
        }
        if (n > 0 && gl == 0) {
            const bool none = K == 0;
            const uint32_t bestk = (~uint32_t(bestkey)) & 0xFFFFu;  // lattice.rs:144 `i as u16`
            b.eos[s] = make_uint4(none ? kNone : eo + bestk, eos_start, uint32_t(int32_t(bestkey >> 32)), 0);
        }
    }
}

// CONN 0: PRUNE and its unpruned twin are separate kernels launched back to back (each keeps its own register
// allocation); the one the batch does not call for — kFlagLongSentence decides, and only the device knows it —
// returns at once.  CONN 1-3 never prune.
// SPACE = the tokenizer ignores spaces: only then can a position carry a skip or the trailing flag.
template <int CONN, bool PRUNE, bool SPACE>
__global__ void __launch_bounds__(32 * kV2Warps, CONN == 0 ? kV2MinBlocks : (32 / kV2Warps)) k_viterbi2(DictView d, Batch b) {
    const uint32_t batch_flags = *b.flags;
    if (batch_flags & kFlagsStandDown) return;
    if (CONN == 0 && PRUNE == ((batch_flags & kFlagLongSentence) != 0)) return;
    __shared__ __align__(16) V2Shared s_warp[kV2Warps];
    const uint32_t sp = uint32_t(__cvta_generic_to_shared(&s_warp[threadIdx.x >> 5]));
    viterbi2_sweep<CONN, PRUNE, SPACE>(d, b, sp);
}

// ---------------------------------------------------------------------------------------------
// Counted runs only: the SURVEY.md §8(d) counters M, T, P, W, walks, E, N and Lattice::add_connid_counts
// (lattice.rs:170-181), read off the finished lattice after K3 and before K4a reuses `ends_meta`.  A thread walks
// the start positions of its sentence as K3 did; a row's size after K3 is the K that K3 saw at that position, since
// only earlier positions append to it.
// ---------------------------------------------------------------------------------------------

// Candidate header of one start position as {cand_ptr, cand_cnt, skip, flags}; the last two live in a side array
// that only the few positions with a skipped space run or the trailing flag ever touch.
__device__ __forceinline__ uint4 load_info(const Batch& b, uint32_t slot) {
    const uint2 i8 = b.info[slot];
    uint4 r = make_uint4(i8.x, i8.y & ~kInfoSpecial, 0, 0);
    if (i8.y & kInfoSpecial) {
        const uint2 ex = b.info_ex[slot];
        r.z = ex.x;
        r.w = ex.y;
    }
    return r;
}

__global__ void __launch_bounds__(256) k_count_lattice(DictView d, Batch b) {
    VBT_STAND_DOWN_IF_REJECTED(b);
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= b.n_sent) return;
    const uint32_t base = b.slot_off[s], n = b.slot_off[s + 1] - 1 - base;
    if (n == 0) return;  // Worker::tokenize returns early on an empty sentence (worker.rs:50-52)
    unsigned long long cE = 0, cN = 2, cM = 0, cT = 0, cP = 0, cW = 0, cWalks = 0;
    uint32_t slot_end = base + n, skip_slot = base;
    for (uint32_t slot = base; slot < slot_end; ++slot) {
        const uint2 m = b.ends_meta[slot];
        const uint32_t K = m.y - m.x;
        // positions inside a skipped space run are never start_node; K == 0: has_previous_node fails
        if (slot < skip_slot || K == 0) continue;  // (lattice.rs:155-157, tokenizer.rs:110-114)
        const uint4 info = load_info(b, slot);
        if (info.w & kInfoTrailing) {  // tokenizer.rs:128-130: EOS starts here
            slot_end = slot;
            break;
        }
        if (info.z) skip_slot = slot + info.z + 1;  // next start_node = start_word + 1 (tokenizer.rs:134-135)
        const uint32_t ncand = info.y;
        cE += (unsigned long long)K * ncand;
        cN += ncand;
        if (b.counters) {  // k_candidates' walks from start_word again, counting (also where ncand == 0)
            const uint32_t sw = slot + info.z;
            WalkStats st{0, 0, 0, 0, 0};
            uint32_t cu = 0;
            if (d.usr_table)
                cu = walk_lexicon<false, true>(d.usr_nodes, d.usr_num_nodes, d.usr_post, b.code_usr, b.groupable, sw,
                                               nullptr, nullptr, st);
            const uint32_t cs = walk_lexicon<false, true>(d.sys_nodes, d.sys_num_nodes, d.sys_post, b.code_sys,
                                                          b.groupable, sw, nullptr, nullptr, st);
            const uint32_t ck =
                gen_unknown<false>(d, sw, b.cinfo[sw], b.groupable[sw], (cu + cs) != 0, nullptr, nullptr);
            cM += st.m;
            cT += st.t;
            cP += st.p;
            cW += st.w + ck;
            cWalks += st.walks;
        }
        if (b.lid_count) {  // Lattice::add_connid_counts (lattice.rs:170-176): one (left, pred.right) edge per predecessor
            for (uint32_t c = 0; c < ncand; ++c)
                atomicAdd(&b.lid_count[b.cand[info.x + c].x & 0xFFFFu], (unsigned long long)K);
            if (ncand)
                for (uint32_t k = 0; k < K; ++k)
                    atomicAdd(&b.rid_count[uint32_t(b.ends_hot[m.x + k].y)], (unsigned long long)ncand);
        }
    }
    // Lattice::insert_eos (lattice.rs:85-101) connects the row of slot_end
    const uint2 me = b.ends_meta[slot_end];
    cE += me.y - me.x;
    if (b.lid_count) {  // lattice.rs:178-181: the EOS edges are counted over ends[len_char]
        const uint2 ml = b.ends_meta[base + n];
        const uint32_t nl = ml.y - ml.x;
        for (uint32_t k = 0; k < nl; ++k) atomicAdd(&b.rid_count[uint32_t(b.ends_hot[ml.x + k].y)], 1ull);
        if (nl) atomicAdd(&b.lid_count[0], (unsigned long long)nl);
    }
    if (b.counters) {
        atomicAdd(&b.counters[kCntE], cE);
        atomicAdd(&b.counters[kCntN], cN);
        atomicAdd(&b.counters[kCntM], cM);
        atomicAdd(&b.counters[kCntT], cT);
        atomicAdd(&b.counters[kCntP], cP);
        atomicAdd(&b.counters[kCntW], cW);
        atomicAdd(&b.counters[kCntWalks], cWalks);
    }
}

// ---------------------------------------------------------------------------------------------
// K4: Lattice::append_top_nodes (lattice.rs:159-168) + Token accessors (token.rs:21-92)
// ---------------------------------------------------------------------------------------------

// K4a walks the best path once (thread / sentence): it counts the tokens and leaves, for the k-th node from the
// end, {lattice entry, end position} in the sentence's own stretch of `ends_meta` (dead after K3, one entry per
// character, and a path has at most one node per character).  After the token-offset scan K4b turns those entries
// into token records with a warp per sentence — the pointer chase is not repeated and the 24-byte records of a
// sentence are written by neighbouring lanes.
__global__ void __launch_bounds__(256) k_backtrack_count(Batch b) {
    VBT_STAND_DOWN_IF_REJECTED(b);
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= b.n_sent) return;
    uint4 e = b.eos[s];
    uint32_t k = 0;
    if (e.x != kNone) {
        const uint32_t base = b.slot_off[s];
        uint32_t cur = e.x, end_node = e.y;
        while (end_node != 0) {
            uint4 c = b.ends_cold[cur];
            b.ends_meta[base + k] = make_uint2(cur, end_node);
            ++k;
            end_node = c.x - base;
            cur = c.y;
        }
    }
    b.n_tok[s] = k;
    if (b.counters && k) atomicAdd(&b.counters[kCntK], (unsigned long long)k);
}

__global__ void __launch_bounds__(256) k_backtrack_write(Batch b) {
    VBT_STAND_DOWN_IF_REJECTED(b);
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
#pragma unroll 1
    for (uint32_t r = 0; r < kSentPerWarp; ++r) {
    const uint32_t s = w * kSentPerWarp + r;
    if (s >= b.n_sent) return;
    const uint32_t base = b.slot_off[s];
    const unsigned long long t0 = b.tok_off[s];
    const uint32_t n = uint32_t(b.tok_off[s + 1] - t0);
    uint2* out = reinterpret_cast<uint2*>(b.tokens);
    for (uint32_t k = lane; k < n; k += 32) {
        const uint2 pe = b.ends_meta[base + k];  // k-th node from the end of the path
        const uint4 c = b.ends_cold[pe.x];
        const uint32_t end_node = pe.y;
        const uint32_t start_node = c.x - base;
        const uint2 i8 = b.info[c.x];
        const uint32_t start_word = start_node + ((i8.y & kInfoSpecial) ? b.info_ex[c.x].x : 0u);  // token.rs:21-24 uses start_word
        const uint2 bytes = make_uint2(b.byte_pos[base + start_word], b.byte_pos[base + end_node]);  // token.rs:28-32
        if (b.compact) {  // opt-in 16-byte record: the character range is a function of the caller's own UTF-8
            reinterpret_cast<uint4*>(b.tokens)[t0 + (n - 1 - k)] = make_uint4(bytes.x, bytes.y, c.z, c.w);
            continue;
        }
        uint2* t = out + (t0 + (n - 1 - k)) * 3;
        t[0] = make_uint2(start_word, end_node);
        t[1] = bytes;
        t[2] = make_uint2(c.z, c.w);  // word_idx, total_cost
    }
    }
}


// ---------------------------------------------------------------------------------------------
// Output stage: the text `tokenize` writes per sentence (tokenize/src/main.rs:83-127):
//   mecab : {surface}\t{feature}\n per token, then EOS\n
//   wakati: surfaces joined by one space, then \n
//   detail: {surface}\t{feature}\tlex_type={:?}\tleft_id={}\tright_id={}\tword_cost={}\ttotal_cost={}\n, then EOS\n
// One warp per sentence.  Pass 1 sizes every token, a scan places it, pass 2 copies bytes.
// ---------------------------------------------------------------------------------------------

__device__ __forceinline__ uint32_t dec_len(uint32_t v) {
    uint32_t n = 1;
    while (v >= 10) {
        v /= 10;
        ++n;
    }
    return n;
}
__device__ __forceinline__ uint32_t dec_len_signed(int32_t v) {
    return v < 0 ? 1 + dec_len(0u - uint32_t(v)) : dec_len(uint32_t(v));
}
__device__ __forceinline__ uint8_t* put_dec(uint8_t* p, uint32_t v) {
    const uint32_t n = dec_len(v);
    for (uint32_t i = n; i-- > 0;) {
        p[i] = uint8_t('0' + v % 10);
        v /= 10;
    }
    return p + n;
}
__device__ __forceinline__ uint8_t* put_dec_signed(uint8_t* p, int32_t v) {
    if (v < 0) {
        *p++ = '-';
        return put_dec(p, 0u - uint32_t(v));
    }
    return put_dec(p, uint32_t(v));
}
__device__ __forceinline__ uint8_t* put_str(uint8_t* p, const char* s) {
    while (*s) *p++ = uint8_t(*s++);
    return p;
}
__device__ __forceinline__ const char* lex_name(uint32_t lex) {  // LexType's Debug names (dictionary.rs:30-40)
    return lex == 0 ? "System" : lex == 1 ? "User" : "Unknown";
}
__device__ __forceinline__ uint32_t lex_name_len(uint32_t lex) { return lex == 0 ? 6 : lex == 1 ? 4 : 7; }

struct TokenText {
    uint32_t start_byte, surf_len, lex, feat_at, feat_len, word_id;
    int32_t total_cost;
};

__device__ __forceinline__ TokenText token_text(const DictView& d, const uint2* __restrict__ tokens, unsigned long long t) {
    const uint2 bytes = tokens[t * 3 + 1], wc = tokens[t * 3 + 2];
    TokenText x;
    x.start_byte = bytes.x;
    x.surf_len = bytes.y - bytes.x;
    x.lex = wc.x >> 30;
    x.word_id = wc.x & 0x3FFFFFFFu;
    x.total_cost = int32_t(wc.y);
    if (x.lex > 2) {  // not a LexType: treated as a word without feature
        x.lex = 2;
        x.word_id = 0x3FFFFFFFu;
    }
    x.feat_at = 0;
    x.feat_len = 0;
    if (x.word_id < d.n_words[x.lex]) {
        const uint32_t a = __ldg(d.feat_off[x.lex] + x.word_id), b = __ldg(d.feat_off[x.lex] + x.word_id + 1);
        x.feat_at = a;
        x.feat_len = b - a;
    }
    return x;
}

__device__ __forceinline__ uint32_t detail_tail_len(const DictView& d, const TokenText& x) {
    const uint2 pr = x.word_id < d.n_words[x.lex] ? __ldg(d.params[x.lex] + x.word_id) : make_uint2(0, 0);
    return 10 + lex_name_len(x.lex) + 9 + dec_len(pr.x & 0xFFFFu) + 10 + dec_len(pr.x >> 16) + 11 +
           dec_len_signed(int32_t(int16_t(pr.y & 0xFFFFu))) + 12 + dec_len_signed(x.total_cost);
}

__global__ void __launch_bounds__(256) k_format_len(DictView d, FormatArgs f) {
    const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= f.n_sent) return;
    const unsigned long long t0 = f.tok_off[s], t1 = f.tok_off[s + 1];
    for (unsigned long long t = t0 + lane; t < t1; t += 32) {
        const TokenText x = token_text(d, f.tokens, t);
        uint32_t len;
        if (f.mode == kOutWakati)
            len = x.surf_len + (t != t0 ? 1u : 0u);
        else if (f.mode == kOutMecab)
            len = x.surf_len + 1 + x.feat_len + 1;
        else
            len = x.surf_len + 1 + x.feat_len + detail_tail_len(d, x) + 1;
        f.tok_len[t] = len;
    }
}

__device__ __forceinline__ void warp_copy(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, uint32_t lane) {
    for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i];
}

__global__ void __launch_bounds__(256) k_format_write(DictView d, FormatArgs f) {
    const uint32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (s >= f.n_sent) return;
    const unsigned long long t0 = f.tok_off[s], t1 = f.tok_off[s + 1];
    const uint32_t term = f.mode == kOutWakati ? 1 : 4;  // "\n" or "EOS\n"
    const unsigned long long shift = (unsigned long long)term * s;  // terminators of the sentences before
    const uint8_t* __restrict__ sent = f.utf8 + f.byte_off[s];
    if (lane == 0) {
        f.text_off[s] = f.tok_text_off[t0] + shift;
        if (s + 1 == f.n_sent) f.text_off[s + 1] = f.tok_text_off[t1] + shift + term;
    }
    for (unsigned long long c = t0; c < t1; c += 32) {
        // lane i stages token c + i; the copies below take one token at a time with all 32 lanes
        const uint32_t cnt = uint32_t(min(32ull, t1 - c));
        TokenText mine = {0, 0, 0, 0, 0, 0, 0};
        unsigned long long at = 0;
        if (lane < cnt) {
            mine = token_text(d, f.tokens, c + lane);
            at = f.tok_text_off[c + lane] + shift;
        }
        for (uint32_t j = 0; j < cnt; ++j) {
            TokenText x;
            x.start_byte = __shfl_sync(kFull, mine.start_byte, j);
            x.surf_len = __shfl_sync(kFull, mine.surf_len, j);
            x.lex = __shfl_sync(kFull, mine.lex, j);
            x.feat_at = __shfl_sync(kFull, mine.feat_at, j);
            x.feat_len = __shfl_sync(kFull, mine.feat_len, j);
            x.word_id = __shfl_sync(kFull, mine.word_id, j);
            x.total_cost = __shfl_sync(kFull, mine.total_cost, j);
            uint8_t* dst = f.text + __shfl_sync(kFull, at, j);
            if (f.mode == kOutWakati) {
                if (c + j != t0) {
                    if (lane == 0) *dst = ' ';
                    ++dst;
                }
                warp_copy(dst, sent + x.start_byte, x.surf_len, lane);
                continue;
            }
            warp_copy(dst, sent + x.start_byte, x.surf_len, lane);
            dst += x.surf_len;
            if (lane == 0) *dst = '\t';
            ++dst;
            if (x.feat_len) warp_copy(dst, d.feat[x.lex] + x.feat_at, x.feat_len, lane);
            dst += x.feat_len;
            if (lane == 0) {
                if (f.mode == kOutDetail) {
                    const uint2 pr = x.word_id < d.n_words[x.lex] ? __ldg(d.params[x.lex] + x.word_id) : make_uint2(0, 0);
                    dst = put_str(dst, "\tlex_type=");
                    dst = put_str(dst, lex_name(x.lex));
                    dst = put_str(dst, "\tleft_id=");
                    dst = put_dec(dst, pr.x & 0xFFFFu);
                    dst = put_str(dst, "\tright_id=");
                    dst = put_dec(dst, pr.x >> 16);
                    dst = put_str(dst, "\tword_cost=");
                    dst = put_dec_signed(dst, int32_t(int16_t(pr.y & 0xFFFFu)));
                    dst = put_str(dst, "\ttotal_cost=");
                    dst = put_dec_signed(dst, x.total_cost);
                }
                *dst = '\n';
            }
        }
    }
    if (lane == 0) {
        uint8_t* dst = f.text + f.tok_text_off[t1] + shift;
        if (f.mode != kOutWakati) dst = put_str(dst, "EOS");
        *dst = '\n';
    }
}

}  // namespace

void launch_format_len(const DictView& d, const FormatArgs& f, cudaStream_t st) {
    if (!f.n_sent) return;
    k_format_len<<<(f.n_sent + 7) / 8, 256, 0, st>>>(d, f);
}

void launch_format_write(const DictView& d, const FormatArgs& f, cudaStream_t st) {
    if (!f.n_sent) return;
    k_format_write<<<(f.n_sent + 7) / 8, 256, 0, st>>>(d, f);
}

void launch_count_chars(const Batch& b, cudaStream_t st) {
    if (!b.n_sent) return;
    uint32_t blocks = (b.n_sent + 8 * kSentPerWarp - 1) / (8 * kSentPerWarp);
    k_count_chars<<<blocks, 256, 0, st>>>(b);
}

void launch_decode(const DictView& d, const Batch& b, cudaStream_t st) {
    if (!b.n_sent) return;
    uint32_t blocks = (b.n_sent + 8 * kSentPerWarp - 1) / (8 * kSentPerWarp);
    k_decode<<<blocks, 256, 0, st>>>(d, b);
}

void launch_candidates(const DictView& d, const Batch& b, uint32_t max_slots, cudaStream_t st) {
    if (!max_slots) return;
    uint32_t blocks = (max_slots + 255) / 256;
    k_candidates<<<blocks, 256, 0, st>>>(d, b);
}

int launch_viterbi(const DictView& d, const Batch& b, int kernel, cudaStream_t st) {
    if (!b.n_sent) return 0;
    const bool space = d.space_mask != 0;
    const uint32_t per_block = kV2Warps * kV2SentPerWarp;
    const uint32_t blocks = (b.n_sent + per_block - 1) / per_block;
#define VBT_LAUNCH_V2(CONN, PRUNE)                                                  \
    do {                                                                            \
        if (space)                                                                  \
            k_viterbi2<CONN, PRUNE, true><<<blocks, 32 * kV2Warps, 0, st>>>(d, b);  \
        else                                                                        \
            k_viterbi2<CONN, PRUNE, false><<<blocks, 32 * kV2Warps, 0, st>>>(d, b); \
    } while (0)
    int launched = 1;
    if (d.connector_kind == 1) {
        VBT_LAUNCH_V2(1, false);
    } else if (d.connector_kind == 2) {
        VBT_LAUNCH_V2(2, false);
    } else if (kernel == 0 || !d.matrix_window) {  // ConnCol<0> needs the matrix inside one 4 GiB window
        VBT_LAUNCH_V2(3, false);
    } else {  // the pruned kernel and its twin for batches with very long sentences
        VBT_LAUNCH_V2(0, true);
        VBT_LAUNCH_V2(0, false);
        launched = 2;
    }
#undef VBT_LAUNCH_V2
    return launched;
}

void launch_count_lattice(const DictView& d, const Batch& b, cudaStream_t st) {
    if (!b.n_sent) return;
    k_count_lattice<<<(b.n_sent + 255) / 256, 256, 0, st>>>(d, b);
}

void launch_backtrack_count(const Batch& b, cudaStream_t st) {
    if (!b.n_sent) return;
    k_backtrack_count<<<(b.n_sent + 255) / 256, 256, 0, st>>>(b);
}

void launch_backtrack_write(const Batch& b, cudaStream_t st) {
    if (!b.n_sent) return;
    k_backtrack_write<<<(b.n_sent + 8 * kSentPerWarp - 1) / (8 * kSentPerWarp), 256, 0, st>>>(b);  // warps over sentences
}

}  // namespace vbt
