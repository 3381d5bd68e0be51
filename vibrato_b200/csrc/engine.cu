// Device engine of the batched Viterbi tokenizer: HBM workspace + launch sequence (one stream).
#include "engine.hpp"

#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

#include <algorithm>
#include <iterator>
#include <cstring>
#include <string>

#include "device_blob.hpp"
#include "kernels.cuh"

namespace vbt {

const char* const kStageNames =
    "count_chars,scan_slots,decode,candidates,scan_ends,viterbi,backtrack_count,scan_tokens,backtrack_write";

namespace {

void cuda_check(cudaError_t e, const char* what) {
    if (e != cudaSuccess) {
        Status st = (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice) ? kNoDevice : kCuda;
        throw Error(st, std::string(what) + ": " + cudaGetErrorString(e));
    }
}
#define CK(x) cuda_check((x), #x)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    void ensure(size_t bytes, double slack = 1.0) {
        if (bytes <= cap) return;
        if (p) CK(cudaFree(p));
        p = nullptr;
        cap = 0;
        size_t want = size_t(double(bytes) * slack) + 256;
        CK(cudaMalloc(&p, want));
        cap = want;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T* as() const {
        return static_cast<T*>(p);
    }
};

struct Control {  // one small block zeroed per batch and read back once
    unsigned long long pool_ctr;
    unsigned long long n_tokens;
    unsigned long long counters[kNumCounters];
    uint32_t flags;
    uint32_t total_slots;
};

// Output iterator for the row-offset scan: writes {offset, offset} (an empty row) into the 8-byte row metadata so that
// no separate initialisation pass is needed.
struct RowMetaOut {
    uint2* p;
    struct Ref {
        uint2* q;
        __host__ __device__ Ref& operator=(uint32_t v) {
            *q = make_uint2(v, v);
            return *this;
        }
    };
    using iterator_category = std::random_access_iterator_tag;
    using value_type = uint32_t;
    using difference_type = ptrdiff_t;
    using pointer = void;
    using reference = Ref;
    __host__ __device__ Ref operator[](difference_type i) const { return Ref{p + i}; }
    __host__ __device__ Ref operator*() const { return Ref{p}; }
    __host__ __device__ RowMetaOut operator+(difference_type i) const { return RowMetaOut{p + i}; }
};

struct CastU64 {
    __host__ __device__ unsigned long long operator()(uint32_t v) const { return v; }
};

// ConnIdCounter totals += the counts of one finished attempt (see EngineImpl::connid_begin / connid_commit).
__global__ void k_add_u64(unsigned long long* dst, const unsigned long long* src, size_t n) {
    size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) dst[i] += src[i];
}

__global__ void k_publish_totals(const uint32_t* slot_off, const unsigned long long* tok_off, uint32_t n_sent, Control* c) {
    c->total_slots = slot_off[n_sent];
    c->n_tokens = tok_off[n_sent];
}

// Chunked host batches: token offsets of a chunk become global by adding the tokens of all earlier
// chunks (kept in a device-resident running total so the host never has to wait for it).
__global__ void k_add_base(unsigned long long* tok_off, uint32_t n_plus_1, const unsigned long long* base) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_plus_1) tok_off[i] += *base;
}
__global__ void k_bump_base(unsigned long long* base, const Control* c) { *base += c->n_tokens; }
__global__ void k_add_value(unsigned long long* tok_off, uint32_t n_plus_1, unsigned long long base) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_plus_1) tok_off[i] += base;
}

struct Workspace {  // every per-(chunk of a)-batch device array
    DevBuf n_slots, slot_off, eos, n_tok, code_sys, code_usr, cinfo, groupable, byte_pos, info, info_ex, ends_cnt,
        ends_meta, cand, ends_hot, ends_cold, scan_tmp;
    void release() {
        for (DevBuf* b : {&n_slots, &slot_off, &eos, &n_tok, &code_sys, &code_usr, &cinfo, &groupable, &byte_pos, &info,
                          &info_ex, &ends_cnt, &ends_meta, &cand, &ends_hot, &ends_cold, &scan_tmp})
            b->release();
    }
};

struct OutSlot {  // where one (chunk of a) batch leaves its results; two of them alternate in chunked runs
    DevBuf tok_off, tokens, ctrl;
    Control* h_ctrl = nullptr;
    cudaEvent_t ev[kNumStages + 1];
    cudaEvent_t done = nullptr, drained = nullptr;
    uint64_t launches = 0;
};

class EngineImpl final : public Engine {
   public:
    EngineImpl(int device, const uint8_t* host_blob, uint64_t d_blob, uint64_t n_bytes, bool ignore_space,
               uint64_t max_grouping_len)
        : device_(device) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
            throw Error(kNoDevice, "no CUDA device available: the tokenizer has no CPU fallback");
        if (device < 0 || device >= count) throw Error(kInvalidArgument, "device ordinal out of range");
        CK(cudaSetDevice(device));
        CK(cudaStreamCreateWithFlags(&own_stream_, cudaStreamNonBlocking));
        stream_ = own_stream_;
        CK(cudaStreamCreateWithFlags(&in_stream_, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&out_stream_, cudaStreamNonBlocking));
        for (auto& o : out_) {
            for (auto& ev : o.ev) CK(cudaEventCreate(&ev));
            CK(cudaEventCreateWithFlags(&o.done, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&o.drained, cudaEventDisableTiming));
            o.ctrl.ensure(sizeof(Control));
            o.h_ctrl = static_cast<Control*>(pinned_alloc(sizeof(Control)));
        }
        CK(cudaEventCreateWithFlags(&in_done_, cudaEventDisableTiming));
        tok_base_.ensure(8);
        BlobHeader h;
        if (host_blob) {
            if (n_bytes < sizeof(BlobHeader)) throw Error(kInvalidArgument, "dictionary image too small");
            std::memcpy(&h, host_blob, sizeof(h));
        } else {
            if (!d_blob || n_bytes < sizeof(BlobHeader)) throw Error(kInvalidArgument, "dictionary image too small");
            CK(cudaMemcpyAsync(&h, reinterpret_cast<const void*>(d_blob), sizeof(h), cudaMemcpyDeviceToHost, stream_));
            CK(cudaStreamSynchronize(stream_));
        }
        if (h.magic != kBlobMagic || h.total_bytes != n_bytes) throw Error(kInvalidArgument, "not a vibrato_b200 dictionary image");
        if (h.connector_kind == 0 && h.matrix_transposed != 1)
            throw Error(kInvalidArgument, "dictionary image: the connection matrix is not stored transposed");
        // k_viterbi2 addresses the connection matrix with a fixed high address word: the matrix must not cross a
        // 4 GiB boundary.  Where the allocation happens to straddle one, the image is placed again, shifted so that
        // the matrix starts on the boundary (at most one extra matrix of padding).
        const uint64_t m_bytes = h.connector_kind == 0 ? uint64_t(h.num_left) * h.num_right * 2 : 0;
        auto crosses = [&](uint64_t base) {
            return m_bytes && ((base + h.off_matrix) >> 32) != ((base + h.off_matrix + m_bytes - 1) >> 32);
        };
        const bool fits_window = m_bytes <= (1ull << 32);
        uint64_t shift = 0;
        if (host_blob || (fits_window && crosses(d_blob))) {
            blob_own_.ensure(n_bytes);
            if (fits_window && crosses(reinterpret_cast<uint64_t>(blob_own_.p))) {
                blob_own_.release();
                blob_own_.ensure(n_bytes + m_bytes + 512);
                const uint64_t base = reinterpret_cast<uint64_t>(blob_own_.p);
                if (crosses(base)) {  // the boundary lies inside the matrix: less than m_bytes ahead of its start
                    const uint64_t boundary = ((base + h.off_matrix) | 0xFFFFFFFFull) + 1;  // next multiple of 4 GiB
                    shift = (boundary - (base + h.off_matrix) + 255) & ~255ull;  // off_matrix is 256-byte aligned
                }
            }
            uint8_t* dst = static_cast<uint8_t*>(blob_own_.p) + shift;
            if (host_blob)
                CK(cudaMemcpyAsync(dst, host_blob, n_bytes, cudaMemcpyHostToDevice, stream_));
            else
                CK(cudaMemcpyAsync(dst, reinterpret_cast<const void*>(d_blob), n_bytes, cudaMemcpyDeviceToDevice, stream_));
            blob_ = dst;
        } else {
            blob_ = reinterpret_cast<const uint8_t*>(d_blob);
        }
        CK(cudaStreamSynchronize(stream_));
        dv_.matrix_window = (m_bytes && fits_window && !crosses(reinterpret_cast<uint64_t>(blob_))) ? 1 : 0;
        dv_.chr2inf = reinterpret_cast<const uint32_t*>(blob_ + h.off_chr2inf);
        dv_.chr2inf_len = h.chr2inf_len;
        dv_.sys_table = reinterpret_cast<const uint32_t*>(blob_ + h.off_sys_table);
        dv_.sys_table_len = h.sys_table_len;
        dv_.sys_nodes = reinterpret_cast<const uint4*>(blob_ + h.off_sys_nodes);
        dv_.sys_num_nodes = h.sys_num_nodes;
        dv_.sys_post = reinterpret_cast<const uint4*>(blob_ + h.off_sys_post);
        if (h.has_user) {
            dv_.usr_table = reinterpret_cast<const uint32_t*>(blob_ + h.off_usr_table);
            dv_.usr_table_len = h.usr_table_len;
            dv_.usr_nodes = reinterpret_cast<const uint4*>(blob_ + h.off_usr_nodes);
            dv_.usr_num_nodes = h.usr_num_nodes;
            dv_.usr_post = reinterpret_cast<const uint4*>(blob_ + h.off_usr_post);
        } else {
            dv_.usr_table = nullptr;
            dv_.usr_table_len = 0;
            dv_.usr_nodes = nullptr;
            dv_.usr_num_nodes = 0;
            dv_.usr_post = nullptr;
        }
        dv_.unk_off = reinterpret_cast<const uint32_t*>(blob_ + h.off_unk_off);
        dv_.unk_ent = reinterpret_cast<const uint2*>(blob_ + h.off_unk_ent);
        dv_.matrix = reinterpret_cast<const int16_t*>(blob_ + h.off_matrix);
        dv_.num_right = h.num_right;
        dv_.conn_stride_left = 1;
        dv_.conn_stride_right = h.num_left;
        dv_.connector_kind = h.connector_kind;
        for (int li = 0; li < 3; ++li) {
            dv_.feat_off[li] = reinterpret_cast<const uint32_t*>(blob_ + h.off_feat_off[li]);
            dv_.feat[li] = blob_ + h.off_feat[li];
            dv_.params[li] = reinterpret_cast<const uint2*>(blob_ + h.off_params[li]);
            dv_.n_words[li] = h.n_words[li];
        }
        dv_.right_conn = dv_.left_conn = nullptr;
        if (h.connector_kind == 1 || h.connector_kind == 2) {
            dv_.right_feats = reinterpret_cast<const uint32_t*>(blob_ + h.off_right_feats);
            dv_.left_feats = reinterpret_cast<const uint32_t*>(blob_ + h.off_left_feats);
            dv_.feat_T = h.feat_T;
            dv_.sc_bases = reinterpret_cast<const uint32_t*>(blob_ + h.off_bases);
            dv_.sc_checks = reinterpret_cast<const uint32_t*>(blob_ + h.off_checks);
            dv_.sc_costs = reinterpret_cast<const int32_t*>(blob_ + h.off_costs);
            dv_.n_bases = h.n_bases;
            dv_.n_checks = h.n_checks;
            if (h.connector_kind == 2) {
                if (h.feat_T != 8) throw Error(kDecode, "dual connector image: the raw term must be 8 lanes wide");
                dv_.num_right = h.m_num_right;
                dv_.right_conn = reinterpret_cast<const uint16_t*>(blob_ + h.off_right_conn);
                dv_.left_conn = reinterpret_cast<const uint16_t*>(blob_ + h.off_left_conn);
            }
        } else if (h.connector_kind != 0) {
            throw Error(kUnsupported, "dictionary image with an unknown connector kind");
        }
        num_left_ = h.num_left;
        num_right_ = h.num_right;
        left_ids_.resize(h.num_left);
        right_ids_.resize(h.num_right);
        CK(cudaMemcpy(left_ids_.data(), blob_ + h.off_left_ids, size_t(h.num_left) * 2, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(right_ids_.data(), blob_ + h.off_right_ids, size_t(h.num_right) * 2, cudaMemcpyDeviceToHost));
        if (ignore_space) {  // Tokenizer::ignore_space tokenizer.rs:42-55
            if (h.space_cate_id < 0)
                throw Error(kInvalidArgument, "dict: SPACE is not defined in the input dictionary (i.e., char.def).");
            dv_.space_mask = 1u << h.space_cate_id;
        } else {
            dv_.space_mask = 0;
        }
        dv_.max_grouping = max_grouping_len ? max_grouping_len : ~0ull;  // tokenizer.rs:67-74
        std::memset(stage_ms_, 0, sizeof(stage_ms_));
        std::memset(counters_, 0, sizeof(counters_));
    }

    ~EngineImpl() override {
        cudaSetDevice(device_);
        cudaStreamSynchronize(stream_);
        cudaStreamSynchronize(in_stream_);
        cudaStreamSynchronize(out_stream_);
        for (auto& o : out_) {
            o.tok_off.release();
            o.tokens.release();
            o.ctrl.release();
            pinned_free(o.h_ctrl);
            for (auto& ev : o.ev) cudaEventDestroy(ev);
            cudaEventDestroy(o.done);
            cudaEventDestroy(o.drained);
        }
        for (int i = 0; i < kRingSlots; ++i) {
            if (ring_[i]) pinned_free(ring_[i]);
            if (ring_ev_[i]) cudaEventDestroy(ring_ev_[i]);
        }
        cudaEventDestroy(in_done_);
        cudaStreamDestroy(in_stream_);
        cudaStreamDestroy(out_stream_);
        tok_base_.release();
        for (auto* b : {&blob_own_, &in_utf8_, &in_off_, &connid_, &connid_try_, &fmt_len_, &fmt_off_, &fmt_text_off_, &fmt_text_}) b->release();
        ws_.release();
        for (auto& r : pool_) {
            pinned_free(r->tok_off);
            pinned_free(r->tokens);
            pinned_free(r->text_off);
            pinned_free(r->text);
            delete r;
        }
        cudaStreamDestroy(own_stream_);
    }

    void set_counting(bool on) override { counting_ = on; }
    void set_option(const std::string& name, long long value) override {
        if (name == "connid_counting") {
            // Worker::init_connid_counter (worker.rs:77-83) when switched on; every batch tokenised
            // while it is on is followed by update_connid_counts (worker.rs:90-93)
            cudaStreamSynchronize(stream_);
            connid_on_ = value != 0;
            if (connid_on_) {
                connid_.ensure((size_t(num_left_) + num_right_) * 8);
                connid_try_.ensure((size_t(num_left_) + num_right_) * 8);
                CK(cudaMemset(connid_.p, 0, (size_t(num_left_) + num_right_) * 8));
            }
        } else if (name == "compact_tokens") {
            // 16-byte token records {start_byte, end_byte, word_idx, total_cost}: a third less to bring back over PCIe;
            // the character range of a token is recomputed by the caller from its own UTF-8 (vbt_result_view_compact)
            if (value != 0 && output_mode_ != kOutNone) throw Error(kInvalidArgument, "compact_tokens and output_mode exclude each other");
            cudaStreamSynchronize(stream_);
            tok_bytes_ = value ? 16 : 24;
        } else if (name == "output_mode") {
            if (value < 0 || value > 3) throw Error(kInvalidArgument, "output_mode must be 0 (off), 1 mecab, 2 wakati or 3 detail");
            if (value != 0 && tok_bytes_ != 24) throw Error(kInvalidArgument, "compact_tokens and output_mode exclude each other");
            output_mode_ = uint32_t(value);
        } else if (name == "chunk_sentences") {
            if (value < 0 || value > 0x7FFFFFFF) throw Error(kInvalidArgument, "chunk_sentences out of range");
            chunk_sentences_ = uint32_t(value);  // 0 disables the chunked host pipeline
        } else if (name == "pool_estimate_permille") {
            // candidates expected per input byte (x 1000): the pool is sized from it and a batch that overflows
            // the pool is re-run with the exact size.  Tests set it low to walk that path.
            if (value < 1 || value > 1000000) throw Error(kInvalidArgument, "pool_estimate_permille out of range");
            cand_per_byte_ = double(value) / 1000.0;
        } else if (name == "chars_estimate_permille") {
            // characters expected per input byte (x 1000) for sizing the per-character launches; tests set it low
            if (value < 1 || value > 1000) throw Error(kInvalidArgument, "chars_estimate_permille out of range");
            chars_per_byte_ = double(value) / 1000.0;
        } else if (name == "viterbi_kernel") {
            if (value < 0 || value > 1) throw Error(kInvalidArgument, "viterbi_kernel must be 0 or 1");
            viterbi_kernel_ = int(value);
        } else if (name == "counting") {
            counting_ = value != 0;
        } else {
            throw Error(kInvalidArgument, "unknown option: " + name);
        }
    }
    void set_stream(uint64_t stream) override {
        cudaStreamSynchronize(stream_);
        stream_ = stream ? reinterpret_cast<cudaStream_t>(stream) : own_stream_;
    }
    const float* stage_ms() const override { return stage_ms_; }
    uint64_t launch_count() const override { return launches_; }
    const uint64_t* counters() const override { return counters_; }
    void connid_counts(uint64_t* lid, uint64_t* rid, uint32_t* num_left, uint32_t* num_right) override {
        if (num_left) *num_left = num_left_;
        if (num_right) *num_right = num_right_;
        if (!lid || !rid) return;
        if (!connid_.p) throw Error(kInvalidArgument, "connid counting was never switched on");
        CK(cudaSetDevice(device_));
        std::vector<unsigned long long> raw(size_t(num_left_) + num_right_);
        CK(cudaMemcpy(raw.data(), connid_.p, raw.size() * 8, cudaMemcpyDeviceToHost));
        for (uint32_t i = 0; i < num_left_; ++i) lid[left_ids_[i]] = raw[i];
        for (uint32_t i = 0; i < num_right_; ++i) rid[right_ids_[i]] = raw[num_left_ + i];
    }

    void run_device(uint64_t d_utf8, uint64_t d_byte_off, uint64_t n_sent, uint64_t n_bytes, uint64_t* d_tok_off,
                    uint64_t* d_tokens, uint64_t* n_tokens) override {
        CK(cudaSetDevice(device_));
        check_size(n_sent, n_bytes);
        run_whole(reinterpret_cast<const uint8_t*>(d_utf8), reinterpret_cast<const unsigned long long*>(d_byte_off),
                  uint32_t(n_sent), n_bytes);
        *d_tok_off = reinterpret_cast<uint64_t>(out_[0].tok_off.p);
        *d_tokens = reinterpret_cast<uint64_t>(out_[0].tokens.p);
        *n_tokens = out_[0].h_ctrl->n_tokens;
    }

    // Host path.  Large batches are cut into chunks that flow through three streams: the H2D copy of
    // chunk i+1 and the D2H copy of chunk i-1 overlap the kernels of chunk i (PCIe is full duplex).
    HostResult* run_host(const char* utf8, const uint64_t* byte_off, uint64_t n_sent64) override {
        CK(cudaSetDevice(device_));
        // offsets may start anywhere in the caller's buffer; ship only the used window
        const uint64_t first = n_sent64 ? byte_off[0] : 0;
        const uint64_t n_bytes = n_sent64 ? byte_off[n_sent64] - first : 0;
        check_size(n_sent64, n_bytes);
        const uint32_t n_sent = uint32_t(n_sent64);
        in_utf8_.ensure(n_bytes + 16, 1.25);
        in_off_.ensure((size_t(n_sent) + 1) * 8, 1.25);
        const uint64_t* off = byte_off;
        if (first != 0) {
            rebased_.resize(size_t(n_sent) + 1);
            for (uint64_t i = 0; i <= n_sent; ++i) rebased_[i] = byte_off[i] - first;
            off = rebased_.data();
        }
        const uint8_t* d_utf8 = in_utf8_.as<uint8_t>();
        const unsigned long long* d_off = in_off_.as<unsigned long long>();
        const bool utf8_pinned = n_bytes == 0 || is_pinned(utf8 + first);
        const bool off_pinned = off != byte_off || is_pinned(byte_off);  // rebased_ is ours (pageable, small)
        staged_bytes_ = 0;
        const uint32_t chunk = chunk_sentences_;
        // the output stage formats the whole batch at once from the device-resident tokens
        const bool chunked = chunk > 0 && n_sent > chunk + chunk / 2 && output_mode_ == kOutNone;
        for (int attempt = 0;; ++attempt) {
            if (!chunked) {
                h2d(in_off_.p, off, (size_t(n_sent) + 1) * 8, stream_, off_pinned && off == byte_off);
                h2d(in_utf8_.p, utf8 + first, n_bytes, stream_, utf8_pinned);
                if (n_bytes <= kEagerBytes && output_mode_ == kOutNone) {
                    // Small batches (a per-sentence Worker loop ends up here) are all latency: the result copies are
                    // queued behind the kernels with an upper bound for the token count (a token spans >= 1 byte), so
                    // that the call makes ONE host synchronisation instead of two.
                    HostResult* r = acquire(n_sent, n_bytes);
                    eager_sink_ = r;
                    try {
                        run_whole(d_utf8, d_off, n_sent, n_bytes);
                    } catch (...) {
                        eager_sink_ = nullptr;
                        release(r);
                        throw;
                    }
                    eager_sink_ = nullptr;
                    r->n_tokens = out_[0].h_ctrl->n_tokens;
                    r->has_text = false;
                    return r;
                }
                run_whole(d_utf8, d_off, n_sent, n_bytes);
                OutSlot& o = out_[0];
                HostResult* r = acquire(n_sent, o.h_ctrl->n_tokens);
                CK(cudaMemcpyAsync(r->tok_off, o.tok_off.p, (size_t(n_sent) + 1) * 8, cudaMemcpyDeviceToHost, stream_));
                if (r->n_tokens) CK(cudaMemcpyAsync(r->tokens, o.tokens.p, r->n_tokens * tok_bytes_, cudaMemcpyDeviceToHost, stream_));
                r->has_text = false;
                if (output_mode_ != kOutNone) format_text(d_utf8, d_off, n_sent, o, r);
                CK(cudaStreamSynchronize(stream_));
                return r;
            }
            // ---- chunked, pipelined -------------------------------------------------------------
            // Chunk plan: a small first chunk (its H2D copy is the pipeline's fill), then halving sizes
            // down to a small last chunk (its D2H copy is the drain); big middle chunks keep the
            // kernels efficient.
            std::vector<uint32_t> bounds{0};
            {
                const uint32_t lo = std::max<uint32_t>(1024, chunk / 2);
                bounds.push_back(std::min(n_sent, lo));
                while (bounds.back() < n_sent) {
                    uint32_t rest = n_sent - bounds.back();
                    uint32_t take = rest <= lo + lo / 2 ? rest : std::max(lo, rest / 2);
                    bounds.push_back(bounds.back() + take);
                }
            }
            const uint32_t n_chunks = uint32_t(bounds.size()) - 1;
            uint64_t max_chunk_bytes = 0;
            uint32_t max_chunk_sent = 0;
            for (uint32_t c = 0; c < n_chunks; ++c) {
                max_chunk_bytes = std::max(max_chunk_bytes, off[bounds[c + 1]] - off[bounds[c]]);
                max_chunk_sent = std::max(max_chunk_sent, bounds[c + 1] - bounds[c]);
            }
            ensure_workspace(ws_, max_chunk_sent, max_chunk_bytes);  // sized once: no cudaMalloc in the pipeline
            for (auto& o : out_) {
                o.tok_off.ensure((size_t(max_chunk_sent) + 1) * 8, 1.25);
                o.tokens.ensure(size_t(max_chunk_bytes) * 24 + 24, 1.25);
            }
            // a pinned result sized from the learned tokens-per-byte ratio (grown below if short)
            HostResult* r = acquire(n_sent, uint64_t(double(n_bytes) * tok_per_byte_) + 1024);
            CK(cudaMemsetAsync(tok_base_.p, 0, 8, stream_));
            connid_begin(stream_);
            h2d(in_off_.p, off, (size_t(n_sent) + 1) * 8, stream_, off_pinned && off == byte_off);
            CK(cudaEventRecord(in_done_, stream_));
            CK(cudaStreamWaitEvent(in_stream_, in_done_, 0));
            std::memset(stage_ms_, 0, sizeof(stage_ms_));
            std::memset(counters_, 0, sizeof(counters_));
            launches_ = 0;
            uint64_t tok_total = 0;
            bool overflow = false, bad_utf8 = false, bad_offsets = false, slots_overflow = false;
            uint64_t slots_seen = 0;
            batch_total_bytes_ = n_bytes;
            std::vector<cudaEvent_t>& h2d_ev = h2d_events(n_chunks);
            auto issue_h2d = [&](uint32_t c) {
                uint32_t s0 = bounds[c], s1 = bounds[c + 1];
                uint64_t b0 = off[s0], b1 = off[s1];
                h2d(in_utf8_.as<uint8_t>() + b0, utf8 + first + b0, b1 - b0, in_stream_, utf8_pinned);
                CK(cudaEventRecord(h2d_ev[c], in_stream_));
            };
            // pinned input: every H2D copy is queued up front on its own stream.  Pageable input is staged by
            // this thread, one chunk ahead of the kernels (the staging of chunk c + 1 overlaps the kernels of c).
            if (utf8_pinned)
                for (uint32_t c = 0; c < n_chunks; ++c) issue_h2d(c);
            else
                issue_h2d(0);
            auto drain = [&](uint32_t c) {  // wait for chunk c's kernels, then queue its D2H copies
                OutSlot& o = out_[c & 1];
                uint32_t s0 = bounds[c], s1 = bounds[c + 1];
                CK(cudaEventSynchronize(o.done));
                if (o.h_ctrl->flags & kFlagUtf8Error) bad_utf8 = true;
                if (o.h_ctrl->flags & kFlagBadOffsets) bad_offsets = true;
                if (o.h_ctrl->flags & kFlagPoolOverflow) overflow = true;
                if (o.h_ctrl->flags & kFlagSlotsOverflow) overflow = slots_overflow = true;
                slots_seen += o.h_ctrl->total_slots;
                for (int i = 0; i < kNumStages; ++i) {
                    float ms = 0;
                    CK(cudaEventElapsedTime(&ms, o.ev[i], o.ev[i + 1]));
                    stage_ms_[i] += ms;
                }
                launches_ += o.launches;
                if (counting_)
                    for (int i = 0; i < kNumCounters; ++i) counters_[i] += o.h_ctrl->counters[i];
                pool_need_ = std::max<uint64_t>(pool_need_, o.h_ctrl->pool_ctr);
                const uint64_t nt = o.h_ctrl->n_tokens;
                if (!overflow && !bad_utf8 && !bad_offsets) {
                    if ((tok_total + nt) * tok_bytes_ > r->cap_tok) {  // rare: grow the pinned buffer, keep what is there
                        CK(cudaStreamSynchronize(out_stream_));
                        size_t cap = size_t(double((tok_total + nt) * 24) * 1.5) + 4096;
                        void* bigger = pinned_alloc(cap);
                        std::memcpy(bigger, r->tokens, tok_total * tok_bytes_);
                        pinned_free(r->tokens);
                        r->tokens = bigger;
                        r->cap_tok = cap;
                    }
                    const bool last = s1 == n_sent;
                    CK(cudaMemcpyAsync(r->tok_off + s0, o.tok_off.p, (size_t(s1 - s0) + (last ? 1 : 0)) * 8,
                                       cudaMemcpyDeviceToHost, out_stream_));
                    if (nt)
                        CK(cudaMemcpyAsync(static_cast<uint8_t*>(r->tokens) + tok_total * tok_bytes_, o.tokens.p, nt * tok_bytes_,
                                           cudaMemcpyDeviceToHost, out_stream_));
                }
                CK(cudaEventRecord(o.drained, out_stream_));
                tok_total += nt;
            };
            pool_need_ = 0;
            for (uint32_t c = 0; c < n_chunks; ++c) {
                OutSlot& o = out_[c & 1];
                uint32_t s0 = bounds[c], s1 = bounds[c + 1];
                CK(cudaStreamWaitEvent(stream_, h2d_ev[c], 0));
                if (c >= 2) CK(cudaStreamWaitEvent(stream_, o.drained, 0));  // slot reused: its D2H must be done
                enqueue(ws_, stream_, d_utf8, d_off + s0, s1 - s0, off[s1] - off[s0], o, tok_base_.as<unsigned long long>());
                if (!utf8_pinned && c + 1 < n_chunks) issue_h2d(c + 1);
                if (c >= 1) drain(c - 1);
            }
            drain(n_chunks - 1);
            CK(cudaStreamSynchronize(out_stream_));
            CK(cudaStreamSynchronize(in_stream_));
            CK(cudaStreamSynchronize(stream_));
            if (bad_offsets) {
                release(r);
                throw Error(kInvalidArgument, "byte_offsets must be non-decreasing and end within the input buffer");
            }
            if (bad_utf8) {
                release(r);
                throw Error(kUtf8, "stream did not contain valid UTF-8");
            }
            if (overflow) {
                release(r);
                if (attempt >= 3) throw Error(kInternal, "candidate pool overflow persists");
                if (slots_overflow) chars_per_byte_ = 1.0;
                cand_per_byte_ = std::max(cand_per_byte_ * 1.5, double(pool_need_) / double(std::max<uint64_t>(1, max_chunk_bytes)) * 1.2);
                continue;
            }
            if (max_chunk_bytes)
                cand_per_byte_ = std::max(0.25, double(pool_need_) / double(max_chunk_bytes) * 1.25);
            if (n_bytes) tok_per_byte_ = std::max(0.02, double(tok_total) / double(n_bytes) * 1.1);
            if (n_bytes) chars_per_byte_ = std::min(1.0, double(slots_seen - n_sent) / double(n_bytes) * 1.10);
            connid_commit(stream_);
            r->n_tokens = tok_total;
            return r;
        }
    }

    void release(HostResult* r) override {
        if (r) pool_free_.push_back(r);
    }

    // ---- shard-level entry points (multi_engine.cu) -------------------------------------------------
    uint64_t run_shard(const char* utf8, const uint64_t* byte_off, uint64_t n_sent64, int src_device) override {
        CK(cudaSetDevice(device_));
        const uint64_t first = n_sent64 ? byte_off[0] : 0;
        const uint64_t n_bytes = n_sent64 ? byte_off[n_sent64] - first : 0;
        check_size(n_sent64, n_bytes);
        const uint32_t n_sent = uint32_t(n_sent64);
        in_utf8_.ensure(n_bytes + 16, 1.25);
        in_off_.ensure((size_t(n_sent) + 1) * 8, 1.25);
        const uint64_t* off = byte_off;
        if (first != 0) {
            rebased_.resize(size_t(n_sent) + 1);
            for (uint64_t i = 0; i <= n_sent; ++i) rebased_[i] = byte_off[i] - first;
            off = rebased_.data();
        }
        h2d(in_off_.p, off, (size_t(n_sent) + 1) * 8, stream_, off == byte_off && is_pinned(byte_off));
        if (n_bytes) {
            if (src_device >= 0 && src_device != device_)
                CK(cudaMemcpyPeerAsync(in_utf8_.p, device_, utf8 + first, src_device, n_bytes, stream_));
            else if (src_device >= 0)
                CK(cudaMemcpyAsync(in_utf8_.p, utf8 + first, n_bytes, cudaMemcpyDeviceToDevice, stream_));
            else
                h2d(in_utf8_.p, utf8 + first, n_bytes, stream_, is_pinned(utf8 + first));
        }
        run_whole(in_utf8_.as<uint8_t>(), in_off_.as<unsigned long long>(), n_sent, n_bytes);
        shard_n_sent_ = n_sent;
        return out_[0].h_ctrl->n_tokens;
    }
    void rebase_shard(uint64_t tok_base) override {
        CK(cudaSetDevice(device_));
        if (tok_base)
            k_add_value<<<(shard_n_sent_ + 256) / 256, 256, 0, stream_>>>(out_[0].tok_off.as<unsigned long long>(),
                                                                         shard_n_sent_ + 1, tok_base);
        CK(cudaStreamSynchronize(stream_));
    }
    void fetch_shard(uint64_t* h_tok_off, void* h_tokens, uint64_t tok_base, bool last) override {
        CK(cudaSetDevice(device_));
        OutSlot& o = out_[0];
        if (tok_base)
            k_add_value<<<(shard_n_sent_ + 256) / 256, 256, 0, stream_>>>(o.tok_off.as<unsigned long long>(), shard_n_sent_ + 1,
                                                                         tok_base);
        CK(cudaMemcpyAsync(h_tok_off, o.tok_off.p, (size_t(shard_n_sent_) + (last ? 1 : 0)) * 8, cudaMemcpyDeviceToHost, stream_));
        if (o.h_ctrl->n_tokens)
            CK(cudaMemcpyAsync(h_tokens, o.tokens.p, o.h_ctrl->n_tokens * tok_bytes_, cudaMemcpyDeviceToHost, stream_));
        CK(cudaStreamSynchronize(stream_));
    }
    void shard_outputs(uint64_t* d_tok_off, uint64_t* d_tokens) const override {
        *d_tok_off = reinterpret_cast<uint64_t>(out_[0].tok_off.p);
        *d_tokens = reinterpret_cast<uint64_t>(out_[0].tokens.p);
    }
    int device() const override { return device_; }
    uint32_t token_bytes() const override { return tok_bytes_; }
    std::string describe() const override {
        return "{\"devices\": [" + std::to_string(device_) + "], \"dictionary_transport\": \"single device\", \"token_gather\": \"none\"}";
    }

   private:
    // Host -> device copy of caller memory.  Pinned (page-locked) memory goes straight to the copy engine; pageable
    // memory is staged through a small ring of pinned buffers owned by the engine, so that the copy stays
    // asynchronous and runs at PCIe speed instead of falling back to the driver's synchronous bounce path.
    static bool is_pinned(const void* p) {
        cudaPointerAttributes a{};
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
    }
    void h2d(void* dst, const void* src, size_t bytes, cudaStream_t st, bool src_pinned) {
        if (!bytes) return;
        if (src_pinned) {
            CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
            return;
        }
        if (!ring_[0]) {
            for (int i = 0; i < kRingSlots; ++i) {
                ring_[i] = static_cast<uint8_t*>(pinned_alloc(kRingBytes));
                CK(cudaEventCreateWithFlags(&ring_ev_[i], cudaEventDisableTiming));
            }
        }
        for (size_t o = 0; o < bytes; o += kRingBytes) {
            const size_t len = std::min(kRingBytes, bytes - o);
            const int slot = ring_next_;
            ring_next_ = (ring_next_ + 1) % kRingSlots;
            CK(cudaEventSynchronize(ring_ev_[slot]));  // the copy that last used this slot has left it
            std::memcpy(ring_[slot], static_cast<const uint8_t*>(src) + o, len);
            CK(cudaMemcpyAsync(static_cast<uint8_t*>(dst) + o, ring_[slot], len, cudaMemcpyHostToDevice, st));
            CK(cudaEventRecord(ring_ev_[slot], st));
        }
        staged_bytes_ += bytes;
    }

    // One attempt at a batch = connid_begin, its enqueue(s), then connid_commit once it is known to have succeeded.
    void connid_begin(cudaStream_t st) {
        if (connid_on_) CK(cudaMemsetAsync(connid_try_.p, 0, (size_t(num_left_) + num_right_) * 8, st));
    }
    void connid_commit(cudaStream_t st) {
        if (!connid_on_) return;
        const size_t n = size_t(num_left_) + num_right_;
        k_add_u64<<<unsigned((n + 255) / 256), 256, 0, st>>>(connid_.as<unsigned long long>(),
                                                                connid_try_.as<unsigned long long>(), n);
        CK(cudaStreamSynchronize(st));
    }

    void check_size(uint64_t n_sent, uint64_t n_bytes) const {
        // warp-per-sentence kernels derive the sentence from a 32-bit global thread index (>> 5): 2^27 is the bound
        if (n_sent >= 0x07FFFFFFull || n_bytes + n_sent >= 0xFFFFFF00ull)
            throw Error(kInvalidArgument, "batch too large: split it (at most 2^27 sentences / 2^32 characters per call)");
    }

    std::vector<cudaEvent_t>& h2d_events(uint32_t n) {
        while (h2d_ev_.size() < n) {
            cudaEvent_t e;
            CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h2d_ev_.push_back(e);
        }
        return h2d_ev_;
    }

    HostResult* acquire(uint64_t n_sent, uint64_t n_tokens) {
        HostResult* r = nullptr;
        if (!pool_free_.empty()) {
            r = pool_free_.back();
            pool_free_.pop_back();
        } else {
            r = new HostResult();
            pool_.push_back(r);
        }
        if ((n_sent + 1) * 8 > r->cap_off) {
            pinned_free(r->tok_off);
            r->cap_off = size_t(double((n_sent + 1) * 8) * 1.25) + 64;
            r->tok_off = static_cast<uint64_t*>(pinned_alloc(r->cap_off));
        }
        if (n_tokens * 24 > r->cap_tok) {
            pinned_free(r->tokens);
            r->cap_tok = size_t(double(n_tokens * 24) * 1.25) + 64;
            r->tokens = pinned_alloc(r->cap_tok);
        }
        r->n_sent = n_sent;
        r->n_tokens = n_tokens;
        r->has_text = false;
        r->token_bytes = tok_bytes_;
        return r;
    }

    // Output stage: size every token's text, scan, copy bytes (k_format_len / k_format_write), D2H into `r`.
    void format_text(const uint8_t* d_utf8, const unsigned long long* d_off, uint32_t n_sent, OutSlot& o, HostResult* r) {
        const uint64_t n_tok = r->n_tokens;
        fmt_len_.ensure((n_tok + 1) * 4, 1.25);
        fmt_off_.ensure((n_tok + 1) * 8, 1.25);
        fmt_text_off_.ensure((size_t(n_sent) + 1) * 8, 1.25);
        FormatArgs f{};
        f.utf8 = d_utf8;
        f.byte_off = d_off;
        f.n_sent = n_sent;
        f.tok_off = o.tok_off.as<unsigned long long>();
        f.tokens = o.tokens.as<uint2>();
        f.tok_len = fmt_len_.as<uint32_t>();
        f.tok_text_off = fmt_off_.as<unsigned long long>();
        f.text_off = fmt_text_off_.as<unsigned long long>();
        f.mode = output_mode_;
        CK(cudaMemsetAsync(fmt_len_.as<uint32_t>() + n_tok, 0, 4, stream_));
        launch_format_len(dv_, f, stream_);
        {
            cub::TransformInputIterator<unsigned long long, CastU64, const uint32_t*> it(fmt_len_.as<uint32_t>(), CastU64());
            size_t tmp = 0;
            CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, it, fmt_off_.as<unsigned long long>(), n_tok + 1, stream_));
            ws_.scan_tmp.ensure(tmp + 1024, 1.5);
            exclusive_scan(ws_, it, fmt_off_.as<unsigned long long>(), n_tok + 1, stream_);
        }
        unsigned long long tok_bytes = 0;
        CK(cudaMemcpyAsync(&tok_bytes, fmt_off_.as<unsigned long long>() + n_tok, 8, cudaMemcpyDeviceToHost, stream_));
        CK(cudaStreamSynchronize(stream_));
        const uint64_t term = output_mode_ == kOutWakati ? 1 : 4;
        const uint64_t total = tok_bytes + term * n_sent;
        fmt_text_.ensure(total + 16, 1.25);
        f.text = fmt_text_.as<uint8_t>();
        if (n_sent == 0) CK(cudaMemsetAsync(fmt_text_off_.p, 0, 8, stream_));
        launch_format_write(dv_, f, stream_);
        launches_ += 2;
        if ((size_t(n_sent) + 1) * 8 > r->cap_text_off) {
            pinned_free(r->text_off);
            r->cap_text_off = size_t(double((size_t(n_sent) + 1) * 8) * 1.25) + 64;
            r->text_off = static_cast<uint64_t*>(pinned_alloc(r->cap_text_off));
        }
        if (total + 1 > r->cap_text) {
            pinned_free(r->text);
            r->cap_text = size_t(double(total + 1) * 1.25) + 64;
            r->text = static_cast<char*>(pinned_alloc(r->cap_text));
        }
        CK(cudaMemcpyAsync(r->text_off, fmt_text_off_.p, (size_t(n_sent) + 1) * 8, cudaMemcpyDeviceToHost, stream_));
        if (total) CK(cudaMemcpyAsync(r->text, fmt_text_.p, total, cudaMemcpyDeviceToHost, stream_));
        r->text_bytes = total;
        r->has_text = true;
    }

    template <typename In, typename Out>
    void exclusive_scan(Workspace& w, In in, Out out, size_t n, cudaStream_t st) {
        size_t cap = w.scan_tmp.cap;  // sized by ensure_workspace
        CK(cub::DeviceScan::ExclusiveSum(w.scan_tmp.p, cap, in, out, n, st));
    }

    // Sizes every workspace array for batches of up to n_sent sentences / n_bytes bytes (upper
    // bounds: characters <= bytes, one sentinel slot per sentence).
    void ensure_workspace(Workspace& w, uint32_t n_sent, uint64_t n_bytes) {
        const size_t ns = size_t(n_sent) + 1;
        w.n_slots.ensure(ns * 4, 1.25);
        w.slot_off.ensure(ns * 4, 1.25);
        w.eos.ensure(ns * 16, 1.25);
        w.n_tok.ensure(ns * 4, 1.25);
        const size_t ms = size_t(n_bytes) + n_sent + 1;
        w.code_sys.ensure(ms * 4, 1.25);
        if (dv_.usr_table) w.code_usr.ensure(ms * 4, 1.25);
        w.cinfo.ensure(ms * 4, 1.25);
        w.groupable.ensure(ms * 4, 1.25);
        w.byte_pos.ensure(ms * 4, 1.25);
        w.info.ensure(ms * 8, 1.25);
        w.info_ex.ensure(ms * 8, 1.25);
        w.ends_cnt.ensure(ms * 4, 1.25);
        w.ends_meta.ensure(ms * 8, 1.25);
        size_t want_cand = std::max<size_t>(1 << 16, size_t(double(n_bytes) * cand_per_byte_) + 4096);
        want_cand = std::min<size_t>(want_cand, 0xFFFFFFF0ull);
        w.cand.ensure(want_cand * 16);
        w.ends_hot.ensure((want_cand + ns) * 8);
        w.ends_cold.ensure((want_cand + ns) * 16);
        size_t tmp = 0;  // cub temp storage for the largest scan of this size
        cub::DeviceScan::ExclusiveSum(nullptr, tmp, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), ms, stream_);
        w.scan_tmp.ensure(tmp + 1024, 1.5);
    }

    // One whole batch from device-resident input into out_[0]; synchronises, retries on pool overflow.
    void run_whole(const uint8_t* d_utf8, const unsigned long long* d_off, uint32_t n_sent, uint64_t n_bytes) {
        OutSlot& o = out_[0];
        batch_total_bytes_ = n_bytes;
        for (int attempt = 0;; ++attempt) {
            ensure_workspace(ws_, n_sent, n_bytes);
            o.tok_off.ensure((size_t(n_sent) + 1) * 8, 1.25);
            o.tokens.ensure(size_t(n_bytes) * 24 + 24, 1.25);  // a token spans >= 1 character >= 1 byte
            connid_begin(stream_);
            enqueue(ws_, stream_, d_utf8, d_off, n_sent, n_bytes, o, nullptr);
            CK(cudaEventSynchronize(o.done));
            CK(cudaGetLastError());
            if (o.h_ctrl->flags & kFlagBadOffsets)
                throw Error(kInvalidArgument, "byte_offsets must be non-decreasing and end within the input buffer");
            if (o.h_ctrl->flags & kFlagUtf8Error)
                throw Error(kUtf8, "stream did not contain valid UTF-8");  // what `stdin.lines()` reports
            if (o.h_ctrl->flags & kFlagSlotsOverflow) {  // more characters per byte than any batch before: hard bound
                if (attempt >= 3) throw Error(kInternal, "slot overflow persists");
                chars_per_byte_ = 1.0;
                continue;
            }
            if (o.h_ctrl->flags & kFlagPoolOverflow) {
                if (attempt >= 3) throw Error(kInternal, "candidate pool overflow persists");
                if (double(o.h_ctrl->pool_ctr) * 1.05 + 4096 >= double(0xFFFFFFF0ull))
                    throw Error(kInvalidArgument, "batch produces more than 2^32 lattice nodes: split it");
                cand_per_byte_ = double(o.h_ctrl->pool_ctr) / double(std::max<uint64_t>(1, n_bytes)) * 1.05 + 1e-3;
                continue;
            }
            if (n_bytes) cand_per_byte_ = std::max(0.25, double(o.h_ctrl->pool_ctr) / double(n_bytes) * 1.15);
            if (n_bytes) chars_per_byte_ = std::min(1.0, double(o.h_ctrl->total_slots - n_sent) / double(n_bytes) * 1.10);
            connid_commit(stream_);
            break;
        }
        for (int i = 0; i < kNumStages; ++i) CK(cudaEventElapsedTime(&stage_ms_[i], o.ev[i], o.ev[i + 1]));
        launches_ = o.launches;
        if (counting_) std::memcpy(counters_, o.h_ctrl->counters, sizeof(counters_));
    }

    // Queues the whole kernel sequence for one (chunk of a) batch on `st`; no host synchronisation.
    // `tok_base` (device) makes the chunk's token offsets global and is advanced by its token count; the chunks of a
    // batch run on one stream, which orders these updates.
    void enqueue(Workspace& w, cudaStream_t st, const uint8_t* d_utf8, const unsigned long long* d_off, uint32_t n_sent,
                 uint64_t n_bytes, OutSlot& o, unsigned long long* tok_base) {
        // characters <= bytes is the hard bound; the per-character launches are sized from the ratio learned on
        // earlier batches (plus slack), and a batch that exceeds it flags itself and is re-run with the hard bound
        const uint32_t hard_slots = uint32_t(n_bytes + n_sent);
        const uint32_t max_slots = uint32_t(std::min<uint64_t>(hard_slots, uint64_t(double(n_bytes) * chars_per_byte_) + n_sent + 4096));
        const uint32_t cand_cap = uint32_t(std::min<size_t>(
            w.cand.cap / 16, std::min<size_t>(w.ends_hot.cap / 8 - n_sent - 1, w.ends_cold.cap / 16 - n_sent - 1)));
        Batch b{};
        b.utf8 = d_utf8;
        b.byte_off = d_off;
        b.total_bytes = batch_total_bytes_;
        b.n_sent = n_sent;
        b.launch_slots = max_slots;
        b.n_slots = w.n_slots.as<uint32_t>();
        b.slot_off = w.slot_off.as<uint32_t>();
        b.eos = w.eos.as<uint4>();
        b.n_tok = w.n_tok.as<uint32_t>();
        b.tok_off = o.tok_off.as<unsigned long long>();
        b.code_sys = w.code_sys.as<uint32_t>();
        b.code_usr = w.code_usr.as<uint32_t>();
        b.cinfo = w.cinfo.as<uint32_t>();
        b.groupable = w.groupable.as<uint32_t>();
        b.byte_pos = w.byte_pos.as<uint32_t>();
        b.info = w.info.as<uint2>();
        b.info_ex = w.info_ex.as<uint2>();
        b.ends_cnt = w.ends_cnt.as<uint32_t>();
        b.ends_meta = w.ends_meta.as<uint2>();
        b.cand = w.cand.as<uint4>();
        b.cand_cap = cand_cap;
        b.ends_hot = w.ends_hot.as<int2>();
        b.ends_cold = w.ends_cold.as<uint4>();
        b.tokens = o.tokens.p;
        b.compact = tok_bytes_ == 16 ? 1u : 0u;
        Control* dc = o.ctrl.as<Control>();
        b.pool_ctr = &dc->pool_ctr;
        b.flags = &dc->flags;
        b.counters = counting_ ? dc->counters : nullptr;
        // counts go to a per-attempt scratch: an attempt that ends in a pool overflow or an input error is re-run
        // or dropped, and must not leave its partial counts behind (lattice.rs:170-181 counts a lattice once)
        b.lid_count = connid_on_ ? connid_try_.as<unsigned long long>() : nullptr;
        b.rid_count = connid_on_ ? connid_try_.as<unsigned long long>() + num_left_ : nullptr;

        o.launches = 0;
        CK(cudaMemsetAsync(dc, 0, sizeof(Control), st));
        CK(cudaEventRecord(o.ev[0], st));
        if (n_sent) {
            launch_count_chars(b, st);
            o.launches += 6;  // count_chars, decode, candidates, backtrack_count, backtrack_write, publish (+ viterbi below)
        } else {
            CK(cudaMemsetAsync(b.n_slots, 0, 4, st));
        }
        CK(cudaEventRecord(o.ev[1], st));
        exclusive_scan(w, b.n_slots, b.slot_off, size_t(n_sent) + 1, st);
        CK(cudaEventRecord(o.ev[2], st));
        launch_decode(dv_, b, st);
        CK(cudaEventRecord(o.ev[3], st));
        launch_candidates(dv_, b, max_slots, st);
        CK(cudaEventRecord(o.ev[4], st));
        exclusive_scan(w, b.ends_cnt, RowMetaOut{b.ends_meta}, size_t(max_slots) + 1, st);
        CK(cudaEventRecord(o.ev[5], st));
        o.launches += launch_viterbi(dv_, b, viterbi_kernel_, st);
        if (b.counters || b.lid_count) {
            launch_count_lattice(dv_, b, st);
            ++o.launches;
        }
        CK(cudaEventRecord(o.ev[6], st));
        launch_backtrack_count(b, st);
        CK(cudaEventRecord(o.ev[7], st));
        {
            cub::TransformInputIterator<unsigned long long, CastU64, const uint32_t*> it(b.n_tok, CastU64());
            if (n_sent == 0) CK(cudaMemsetAsync(b.n_tok, 0, 4, st));
            exclusive_scan(w, it, b.tok_off, size_t(n_sent) + 1, st);
        }
        CK(cudaEventRecord(o.ev[8], st));
        launch_backtrack_write(b, st);
        k_publish_totals<<<1, 1, 0, st>>>(b.slot_off, b.tok_off, n_sent, dc);
        if (tok_base) {
            k_add_base<<<(n_sent + 256) / 256, 256, 0, st>>>(b.tok_off, n_sent + 1, tok_base);
            k_bump_base<<<1, 1, 0, st>>>(tok_base, dc);
            o.launches += 2;
        }
        CK(cudaEventRecord(o.ev[9], st));
        CK(cudaMemcpyAsync(o.h_ctrl, dc, sizeof(Control), cudaMemcpyDeviceToHost, st));
        if (eager_sink_) {  // small batch: results leave in the same breath (sized by their upper bound)
            CK(cudaMemcpyAsync(eager_sink_->tok_off, o.tok_off.p, (size_t(n_sent) + 1) * 8, cudaMemcpyDeviceToHost, st));
            if (n_bytes) CK(cudaMemcpyAsync(eager_sink_->tokens, o.tokens.p, size_t(n_bytes) * tok_bytes_, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaEventRecord(o.done, st));
    }

    int device_;
    static constexpr int kRingSlots = 4;
    static constexpr size_t kRingBytes = size_t(4) << 20;
    uint8_t* ring_[kRingSlots] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ring_ev_[kRingSlots] = {nullptr, nullptr, nullptr, nullptr};
    int ring_next_ = 0;
    static constexpr uint64_t kEagerBytes = 16384;
    HostResult* eager_sink_ = nullptr;
    uint64_t staged_bytes_ = 0;  // bytes of pageable caller memory that went through the ring (last batch)
    uint32_t shard_n_sent_ = 0;
    cudaStream_t stream_ = nullptr, own_stream_ = nullptr, in_stream_ = nullptr, out_stream_ = nullptr;
    cudaEvent_t in_done_ = nullptr;
    std::vector<cudaEvent_t> h2d_ev_;
    OutSlot out_[2];
    DevBuf tok_base_;
    uint32_t chunk_sentences_ = 262144;
    uint64_t pool_need_ = 0;
    double tok_per_byte_ = 0.2;
    DictView dv_{};
    const uint8_t* blob_ = nullptr;
    DevBuf blob_own_, in_utf8_, in_off_, connid_, connid_try_;
    bool connid_on_ = false;
    uint32_t num_left_ = 0, num_right_ = 0;
    std::vector<uint16_t> left_ids_, right_ids_;
    Workspace ws_;
    std::vector<HostResult*> pool_, pool_free_;
    std::vector<uint64_t> rebased_;
    double cand_per_byte_ = 4.0;
    double chars_per_byte_ = 1.0;  // learned; 1.0 = the hard bound (every byte a character)
    bool counting_ = false;
    uint32_t output_mode_ = 0;
    uint64_t batch_total_bytes_ = 0;  // size of the input buffer of the batch in flight (bounds check in K1a)
    DevBuf fmt_len_, fmt_off_, fmt_text_off_, fmt_text_;
    uint32_t tok_bytes_ = 24;
    int viterbi_kernel_ = 1;  // 1 = k_viterbi2 with pruning (kernels.cuh)
    float stage_ms_[kNumStages];
    uint64_t launches_ = 0;
    uint64_t counters_[kNumCounters];
};

}  // namespace

std::unique_ptr<Engine> Engine::create(int device, const uint8_t* host_blob, uint64_t d_blob, uint64_t n_bytes,
                                       bool ignore_space, uint64_t max_grouping_len) {
    return std::unique_ptr<Engine>(new EngineImpl(device, host_blob, d_blob, n_bytes, ignore_space, max_grouping_len));
}

void* pinned_alloc(size_t n) {
    void* p = nullptr;
    cuda_check(cudaHostAlloc(&p, n ? n : 1, cudaHostAllocDefault), "cudaHostAlloc");
    return p;
}

void pinned_free(void* p) {
    if (p) cudaFreeHost(p);
}

}  // namespace vbt
