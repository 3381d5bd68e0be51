// Device engine: owns the dictionary image in HBM, the per-batch workspace and the launch sequence.
#pragma once

#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "host_dict.hpp"

namespace vbt {

struct HostResult {  // pinned host memory holding one batch's tokens
    uint64_t n_sent = 0, n_tokens = 0;
    uint64_t* tok_off = nullptr;  // n_sent + 1
    void* tokens = nullptr;       // vbt_token[n_tokens], or vbt_token16[n_tokens] when token_bytes == 16
    uint32_t token_bytes = 24;
    size_t cap_off = 0, cap_tok = 0;
    // output stage ("output_mode" option): the text `tokenize` prints for the batch and where each sentence's
    // part starts (n_sent + 1 offsets); text == nullptr when the stage is off
    uint64_t text_bytes = 0;
    uint64_t* text_off = nullptr;
    char* text = nullptr;
    size_t cap_text_off = 0, cap_text = 0;
    bool has_text = false;
};

constexpr int kNumStages = 9;
extern const char* const kStageNames;  // comma-separated, kNumStages entries

class Engine {
   public:
    // host_blob: packed dictionary image (device_blob.hpp) to upload; or d_blob: an image already
    // resident on `device` (not owned).
    static std::unique_ptr<Engine> create(int device, const uint8_t* host_blob, uint64_t d_blob, uint64_t n_bytes,
                                          bool ignore_space, uint64_t max_grouping_len);
    // One tokenizer over several devices of this node (multi_engine.cu): the image is uploaded to devices[0] and
    // broadcast (NCCL when libnccl.so.2 loads, peer copies otherwise); batches are split by bytes.
    static std::unique_ptr<Engine> create_multi(const std::vector<int>& devices, const uint8_t* host_blob, uint64_t n_bytes,
                                                bool ignore_space, uint64_t max_grouping_len);
    virtual ~Engine() = default;

    // Inputs/outputs in device memory; outputs owned by the engine until the next call.
    virtual void run_device(uint64_t d_utf8, uint64_t d_byte_off, uint64_t n_sent, uint64_t n_bytes,
                            uint64_t* d_tok_off, uint64_t* d_tokens, uint64_t* n_tokens) = 0;
    // Inputs/outputs in host memory (copies inside).
    virtual HostResult* run_host(const char* utf8, const uint64_t* byte_off, uint64_t n_sent) = 0;
    virtual void release(HostResult* r) = 0;

    // Building blocks of the multi-device engine (multi_engine.cu); a single-device caller never needs them.
    // run_shard: host sentences in, tokens left in this device's memory; returns their number (synchronises).
    // With src_device >= 0 `utf8` is a DEVICE address on that device (peer copy over NVLink) while byte_off is
    // still a host array.
    virtual uint64_t run_shard(const char* utf8, const uint64_t* byte_off, uint64_t n_sent, int src_device) = 0;
    // fetch_shard: the last shard's token offsets (+ tok_base, n_sent entries, one more when `last`) and token
    // records into host memory (pinned, or it is slow).
    virtual void fetch_shard(uint64_t* h_tok_off, void* h_tokens, uint64_t tok_base, bool last) = 0;
    // Device addresses of the last shard's token offsets (uint64[n_sent + 1], already + tok_base after
    // rebase_shard) and token records.
    virtual void rebase_shard(uint64_t tok_base) = 0;
    virtual void shard_outputs(uint64_t* d_tok_off, uint64_t* d_tokens) const = 0;
    virtual int device() const = 0;
    virtual uint32_t token_bytes() const = 0;  // 24, or 16 with the "compact_tokens" option
    virtual std::string describe() const = 0;  // JSON: devices, how the dictionary travelled, ...

    virtual void set_counting(bool on) = 0;
    // Knobs: "counting" (0/1), "chunk_sentences", "connid_counting", "output_mode" (0 none, 1 mecab, 2 wakati,
    // 3 detail: run_host also produces HostResult::text).
    virtual void set_option(const std::string& name, long long value) = 0;
    // Launch on a caller-owned CUDA stream (0 restores the engine's own stream).
    virtual void set_stream(uint64_t stream) = 0;
    virtual const float* stage_ms() const = 0;
    virtual uint64_t launch_count() const = 0;
    virtual const uint64_t* counters() const = 0;  // 10 entries, valid after a counted batch
    // ConnIdCounter (mapper.rs:87-104) accumulated since "connid_counting" was switched on, in the
    // dictionary's own connection ids: lid[num_left], rid[num_right].
    virtual void connid_counts(uint64_t* lid, uint64_t* rid, uint32_t* num_left, uint32_t* num_right) = 0;
};

// Restricts the calling thread to the CPUs of the NUMA node `device` is attached to (never beyond the process's
// own affinity mask); a no-op where sysfs does not say.
void pin_thread_to_device_numa_node(int device);

void* pinned_alloc(size_t n);
void pinned_free(void* p);

}  // namespace vbt
