#!/usr/bin/env python3
"""bench.py — sentences/sec of the batched Viterbi tokenizer on B200 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5]    # our arm (CUDA path through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...              # the reference's CPU path on host cores

A "step" = one pass of the hot path over one batch of synthetic sentences.  The default workload (--config 3) is
BASELINE.json configs[2], the one the metric is quoted on: a unidic-cwj-3.1.1-shaped dictionary (876 803 words,
15 626 x 15 388 i16 connection matrix = 459 MiB) and ONE batch of 1 M ~40-character sentences.  No real dictionary
exists in this environment, so both are seeded synthetic data (vibrato_b200/synth.py) — `"data": "synthetic"`.
--config 2 / 4 / 5 select the other BASELINE configurations (ipadic-shaped 100 k; ipadic + user.csv, mixed 8-256
chars, 100 k; unidic-shaped 10 k x 512 chars); they are parity-test cases first and bench lines second
(profiles/r02_bench_config*.json).

With N > 1 (one process per GPU under torchrun) the SAME batch is split over the ranks by bytes — strong scaling,
what BASELINE.json's north_star asks for ("2/4/8-GPU runs split the batch").  Rank 0 packs the dictionary image
once and NCCL-broadcasts it; there is no collective in the data path of `value` / `e2e` (every rank's tokens go
to its own host over its own PCIe link).  `gathered` adds the NVLink route for device-resident consumers: token
counts all-gathered, token records sent to rank 0's GPU with one NCCL all-to-all.  `weak` reports the round-1
style line (every rank a full batch of its own) next to it.

`value`  = sentences/s with the batch already resident in HBM (device-resident C-ABI entry point),
           timed with CUDA events on the launching stream, max over ranks.
`e2e`    = the same metric through vbt_tokenize_batch with pinned HOST buffers: host->device copy of the
           sentences and device->host copy of the token records inside the timed region.
           `e2e.pageable` = the same call on ordinary (pageable) host memory, which the library stages through
           its own pinned ring.
`roofline` is for the dominant kernel (k_viterbi2): algorithmic bytes 2*E + 20*N (SURVEY.md §8d: E connection-cost
           lookups of 2 B, N lattice nodes of 20 B, both from device counters of this very batch) over its
           CUDA-event duration.  The kernel skips lookups that provably cannot win (exact lower-bound pruning,
           DESIGN.md §4); E still counts every edge of the lattice, as the reference evaluates them.
`cpu_baseline` = the oracle (a C restatement of vibrato's Rust path; the Rust toolchain is absent) timed with the
           reference's benchmark protocol body on one host thread, bounded sample.

--dump-outputs DIR writes what the last timed step of `value` returned (the device-resident entry point's token
offsets and token records) as DIR/<name>.npy, so that two builds can be compared output for output on the same
seeded inputs; see dump_outputs() for the files.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "sentences/sec (unidic-cwj-3.1.1, batch 1M) at 1/2/4/8 B200 vs ref CPU"

# BASELINE.json configs (SURVEY.md §8(d) numbering: 2..5; 1 is the single-sentence plumbing case of the tests)
CONFIGS = {
    2: dict(dict="synth-ipadic", batch=100000, corpus={}, user=False, cpu_sample=100000,
            text="batch 100k synthetic ~40-char JA sentences (BASELINE.json configs[1])",
            lens="round(N(40,8^2)) clipped to [8,120]"),
    3: dict(dict="synth-unidic", batch=1000000, corpus={}, user=False, cpu_sample=200000,
            text="batch 1M synthetic ~40-char JA sentences (BASELINE.json configs[2])",
            lens="round(N(40,8^2)) clipped to [8,120]"),
    4: dict(dict="synth-ipadic", batch=100000, corpus=dict(log_uniform=(8, 256), unk_frac=0.15, user_frac=0.05),
            user=True, cpu_sample=100000,
            text="+ user.csv (1000 rows), 100k sentences of mixed 8-256 chars, 15% unknown-word runs, 5% with user "
                 "surfaces (BASELINE.json configs[3])", lens="log-uniform in [8,256]"),
    5: dict(dict="synth-unidic", batch=10000, corpus=dict(fixed_len=512), user=False, cpu_sample=10000,
            text="10k x 512-char sentences: deep lattice, high predecessor fan-in (BASELINE.json configs[4])",
            lens="exactly 512"),
}
STAND_IN = {"synth-unidic": "unidic-cwj-3.1.1", "synth-ipadic": "ipadic-mecab-2.7.0"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Libraries (NCCL prints its version banner) may write to stdout; the contract is ONE JSON line there.
# Everything written to fd 1 during the run is diverted to stderr, the result goes to the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.windows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark(self):
        """Opens / closes a timed window; only samples inside windows are reported."""
        self.windows.append(time.time())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        wins = list(zip(self.windows[0::2], self.windows[1::2]))
        inside = [ln for (t, ln) in self.lines if any(a - 0.05 <= t <= b + 0.15 for a, b in wins)]
        if not inside:  # very short runs: fall back to everything sampled since start()
            inside = [ln for (_, ln) in self.lines]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Threads the CPU arm may really use: the affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0))
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def make_inputs(cfg, rank, need_matrix, seed_rank=0):
    from vibrato_b200 import synth
    t = time.time()
    sd = synth.make_dictionary(cfg["dict"], with_matrix=need_matrix)
    log(f"[rank {rank}] synthetic dictionary {cfg['dict']}: {time.time() - t:.1f}s")
    t = time.time()
    user_csv = synth.make_user_csv(sd) if cfg["user"] else None
    kw = dict(cfg["corpus"])
    if cfg["user"]:
        kw["user_csv"] = user_csv
    utf8, off = synth.make_corpus(sd, cfg["batch"], seed=20260923 + 2 + 1000 * seed_rank, **kw)
    log(f"[rank {rank}] corpus {cfg['batch']} sentences, {len(utf8) / 1e6:.1f} MB: {time.time() - t:.1f}s")
    return sd, user_csv, utf8, off


def device_to_host(ptr, nbytes):
    """Copies nbytes of device memory at ptr (a pointer the library returned) into a numpy uint8 array."""
    import torch

    class View:
        __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}

    if nbytes == 0:
        return np.zeros(0, dtype=np.uint8)
    return torch.as_tensor(View(), device="cuda").cpu().numpy()


DUMP_SEED = 20261017
# Every token covers at least one input byte, so the sample holds at most 900 000 tokens (43.2 MB as 6 float64 fields);
# with the per-sentence counts (<= 16 MB) and the sample's index and offsets (<= 1.1 MB) the files stay under 64 MB.
DUMP_SAMPLE_INPUT_BYTES = 900_000
DUMP_SAMPLE_MAX_SENTENCES = 65536
DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, tok_off, tokens, off):
    """Writes one step's result as float64 / float32 .npy files (every value is exact in its type):

    tokens_per_sentence  float32 [n_sent]   token count of every sentence of the batch (left out above 4 M sentences)
    sentence_index       float64 [S]        a fixed sample of sentences (seeded from DUMP_SEED and the input lengths only)
    tok_offsets          float64 [S + 1]    where each sampled sentence's tokens start in the arrays below
    <field>              float64 [T]        start_char, end_char, start_byte, end_byte, word_idx, total_cost of the
                                            sampled sentences' tokens, in sentence order
    """
    import vibrato_b200 as vb
    n = len(tok_off) - 1
    tok_off = tok_off.astype(np.int64)
    files = {}
    if n <= 4_000_000:
        files["tokens_per_sentence"] = np.diff(tok_off).astype(np.float32)
    order = np.random.default_rng(DUMP_SEED).permutation(n)
    in_bytes = np.cumsum(np.diff(off.astype(np.int64))[order])
    k = min(int(np.searchsorted(in_bytes, DUMP_SAMPLE_INPUT_BYTES, side="right")), DUMP_SAMPLE_MAX_SENTENCES)
    idx = np.sort(order[:k])
    counts = tok_off[idx + 1] - tok_off[idx]
    sample_off = np.concatenate([[0], np.cumsum(counts)])
    rows = np.arange(sample_off[-1]) - np.repeat(sample_off[:-1] - tok_off[idx], counts)
    files["sentence_index"] = idx.astype(np.float64)
    files["tok_offsets"] = sample_off.astype(np.float64)
    for name in vb.TOKEN_DTYPE.names:
        files[name] = tokens[name][rows].astype(np.float64)
    total = sum(a.nbytes for a in files.values())
    assert total <= DUMP_MAX_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in files.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"outputs of the last timed step: {len(files)} arrays, {total / 1e6:.1f} MB -> {out_dir}")


def workload_config(cfg_id, cfg):
    """Identical for both arms (the driver compares them): the CPU arm's bounded sample is part of the text."""
    from vibrato_b200 import synth
    nw, nr, nl, _, _ = synth.SHAPES[cfg["dict"]]
    return {
        "workload": f"{cfg['dict']}: synthetic stand-in for {STAND_IN[cfg['dict']]} ({nw} words, {nl}x{nr} i16 connection "
                    f"matrix = {nl * nr * 2 / 2**20:.0f} MiB); {cfg['text']}; with N GPUs the one batch is split over "
                    f"the GPUs by bytes (strong scaling); the CPU arm (--impl reference, cpu_baseline) times the first "
                    f"{min(cfg['cpu_sample'], cfg['batch'])} sentences of the same batch per step",
        "config_id": cfg_id,
        "dictionary": "synthetic (no real unidic/ipadic in this environment)",
        "batch": cfg["batch"],
        "sentence_len_chars": cfg["lens"],
        "cache": "inputs_exceed_l2 (sentences + lattice workspace touched per step are hundreds of MB to GBs; L2 is 126 MB)",
        "parallelism": "shard-over-sentences, replicated dictionary",
    }


def run_reference(args, cfg_id, cfg, rank, world):
    """The reference's own CPU implementation of the path = the oracle (C restatement; the Rust crate cannot be
    built here), all host threads this process may use, bounded sample per step; a 1-thread figure beside it."""
    if rank != 0:
        return
    from oracle import vibrato_oracle as vo
    sd, user_csv, utf8, off = make_inputs(cfg, 0, True)
    t = time.time()
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    if user_csv is not None:
        od.set_user_csv(user_csv)
    log(f"oracle dictionary build: {time.time() - t:.1f}s")
    threads = host_threads()
    n = min(cfg["cpu_sample"], cfg["batch"])
    sub_off = off[: n + 1]
    for _ in range(args.warmup):
        od.benchmark(utf8, sub_off, n_threads=threads, runs=1)
    secs, nwords = od.benchmark(utf8, sub_off, n_threads=threads, runs=args.steps)
    value = n * args.steps / secs
    n1 = max(1, n // 8)
    od.benchmark(utf8, off[: n1 // 4 + 1], n_threads=1, runs=1)
    secs1, _ = od.benchmark(utf8, off[: n1 + 1], n_threads=1, runs=1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "sentences/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": workload_config(cfg_id, cfg),
        "cpu_baseline": {"value": value, "unit": "sentences/s", "cores": threads, "kind": "port",
                         "one_thread_value": n1 / secs1,
                         "sample": f"{n} sentences x {args.steps} steps on {threads} threads (affinity mask capped by the "
                                   f"cgroup quota; os.cpu_count() = {os.cpu_count()}); one_thread_value = {n1} sentences on "
                                   "1 thread; oracle = C restatement of vibrato 0.5.2 (Rust toolchain absent), protocol body "
                                   "of benchmark/src/main.rs:53-65"},
        "e2e": {"value": value, "unit": "sentences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "n_words": int(nwords),
    }
    emit(line)


def run_ours(args, cfg_id, cfg, rank, world, local_rank):
    import torch
    import vibrato_b200 as vb
    from vibrato_b200._native import check, lib
    import ctypes as C

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the tokenizer has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    lib().vbt_pin_thread_to_device(local_rank)  # host-side copies of this rank stay on the GPU's NUMA node
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    BATCH = cfg["batch"]
    # every rank synthesises the same batch (same seed) and keeps its shard of it
    sd, user_csv, utf8_all, off_all = make_inputs(cfg, rank, rank == 0)
    from vibrato_b200 import distributed as vd
    s0, s1 = vd.shard_by_bytes(off_all, world)[rank]
    n_mine = s1 - s0
    b0, b1 = int(off_all[s0]), int(off_all[s1])
    utf8 = np.ascontiguousarray(utf8_all[b0:b1])
    off = (off_all[s0:s1 + 1] - off_all[s0]).astype(np.uint64)
    n_bytes = int(off[-1])

    # --- dictionary image: rank 0 packs it, everyone else receives it over NCCL ------------------
    t = time.time()
    if rank == 0:
        d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
        if user_csv is not None:
            d.reset_user_lexicon_from_reader(user_csv)
        blob_h = d.pack_blob()
        size = torch.tensor([blob_h.nbytes], dtype=torch.int64, device="cuda")
        log(f"[rank 0] host dictionary + image ({blob_h.nbytes / 2**20:.0f} MiB): {time.time() - t:.1f}s")
    else:
        size = torch.zeros(1, dtype=torch.int64, device="cuda")
    if dist:
        dist.broadcast(size, 0)
    blob = torch.empty(int(size.item()), dtype=torch.uint8, device="cuda")
    if rank == 0:
        blob.copy_(torch.from_numpy(blob_h))
    if dist:
        dist.broadcast(blob, 0)  # the one collective outside the data path: dictionary image over NVLink
    torch.cuda.synchronize()
    h = C.c_void_p()
    check(lib().vbt_tokenizer_new_from_device_blob(blob.data_ptr(), blob.numel(), 0, 0, local_rank, C.byref(h)))
    stream = torch.cuda.current_stream()
    check(lib().vbt_tokenizer_set_stream(h, stream.cuda_stream))
    for opt in ("lanes_per_sentence", "sort_by_length", "chunk_sentences", "dual_stream", "viterbi_kernel"):  # developer overrides
        if os.environ.get("VBT_" + opt.upper()):
            check(lib().vbt_tokenizer_set_option(h, opt.encode(), int(os.environ["VBT_" + opt.upper()])))

    class Inputs:
        def __init__(self, u8, of):
            self.n = len(of) - 1
            self.n_bytes = int(of[-1])
            self.h_utf8 = torch.from_numpy(u8).pin_memory() if len(u8) else torch.zeros(1, dtype=torch.uint8).pin_memory()
            self.h_off = torch.from_numpy(of.astype(np.int64)).pin_memory()
            self.p_utf8 = np.array(u8, copy=True) if len(u8) else np.zeros(1, dtype=np.uint8)  # pageable copies
            self.p_off = np.array(of, dtype=np.uint64, copy=True)
            self.d_utf8 = self.h_utf8.cuda()
            self.d_off = self.h_off.cuda()

    mine = Inputs(utf8, off)
    torch.cuda.synchronize()

    def step_device(inp):
        a, b, n = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib().vbt_tokenize_batch_device(h, inp.d_utf8.data_ptr(), inp.d_off.data_ptr(), inp.n, inp.n_bytes, C.byref(a),
                                              C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def step_host(inp, pageable=False):
        r = C.c_void_p()
        if pageable:
            check(lib().vbt_tokenize_batch(h, inp.p_utf8.ctypes.data, inp.p_off.ctypes.data, inp.n, C.byref(r)))
        else:
            check(lib().vbt_tokenize_batch(h, inp.h_utf8.data_ptr(), inp.h_off.data_ptr(), inp.n, C.byref(r)))
        nt = C.c_uint64()
        check(lib().vbt_result_view(r, None, None, None, C.byref(nt)))
        lib().vbt_result_free(r)
        return nt.value

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def stage_ms():
        ms = (C.c_float * 16)()
        n = C.c_int32()
        check(lib().vbt_last_stage_ms(h, ms, 16, C.byref(n)))
        return np.array([ms[i] for i in range(n.value)], dtype=np.float64)

    def timed(fn, steps, warm):
        """W warm-up calls, then `steps` calls between a barrier + synchronize on both sides; device time by CUDA
        events on the launching stream, max over ranks."""
        for _ in range(warm):
            fn()
        barrier()
        sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1.record(stream)
        barrier()
        sampler.mark()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), out

    stage_names = lib().vbt_stage_names().decode().split(",")

    # one counted batch (outside the timed region): E, N and the whole-path B_alg of this rank's shard
    check(lib().vbt_tokenizer_set_counting(h, 1))
    _, _, n_tokens = step_device(mine)
    cnt = (C.c_uint64 * 10)()
    check(lib().vbt_last_counters(h, cnt))
    cnt = np.array(list(cnt), dtype=np.float64)
    check(lib().vbt_tokenizer_set_counting(h, 0))
    w = np.array([1, 4, 4, 8, 4, 6, 2, 20, 24, 0], dtype=np.float64)
    b_alg_step = float((cnt * w).sum())
    b_alg_viterbi = float(2 * cnt[6] + 20 * cnt[7])
    nl = C.c_uint64()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    W = max(args.warmup, 3)
    stage_acc = np.zeros(len(stage_names))

    def dev_step():
        r = step_device(mine)
        stage_acc[:] += stage_ms()
        return r

    dev_ms, _ = timed(lambda: step_device(mine), 0, W)  # warm-up only
    stage_acc[:] = 0
    dev_ms, last = timed(dev_step, args.steps, 0)
    check(lib().vbt_last_launch_count(h, C.byref(nl)))
    launches_per_step = nl.value
    if args.dump_outputs:  # fetched now: the next call on this tokenizer reuses the result buffers
        p_off, p_tok, n_last = last
        last_tok_off = device_to_host(p_off, (mine.n + 1) * 8).view("<u8")
        last_tokens = device_to_host(p_tok, n_last * vb.TOKEN_DTYPE.itemsize).view(vb.TOKEN_DTYPE)

    # --- e2e: host buffers in, host tokens out (pinned, then pageable) ----------------------------------
    e2e_ms, nt_host = timed(lambda: step_host(mine), args.steps, 2)
    assert nt_host == n_tokens
    e2e_pg_ms, nt_pg = timed(lambda: step_host(mine, pageable=True), args.steps, 2)
    assert nt_pg == n_tokens
    check(lib().vbt_tokenizer_set_option(h, b"compact_tokens", 1))  # opt-in 16-byte records: a third less D2H
    e2e_c_ms, nt_c = timed(lambda: step_host(mine), args.steps, 2)
    assert nt_c == n_tokens
    check(lib().vbt_tokenizer_set_option(h, b"compact_tokens", 0))

    # --- N > 1: the NVLink gather of token records to rank 0, and the weak-scaling line ------------------------
    gathered = weak = None
    if dist:
        def step_gather():
            p_off, p_tok, n = step_device(mine)
            counts = vd.all_gather_counts(n, mine.n, device="cuda")[:, 1]
            # the engine's token records, viewed as 3 x int64 per token (copied out of the engine's buffer)
            mine_rec = torch.empty(n * 3, dtype=torch.int64, device="cuda")
            rt.cudaMemcpyAsync(C.c_void_p(mine_rec.data_ptr()), C.c_void_p(p_tok), C.c_size_t(n * 24), C.c_int(3),
                               C.c_void_p(stream.cuda_stream))
            got = vd.gather_token_records(mine_rec, counts, dst=0)
            return int(got.numel() // 3) if got is not None else 0

        rt = C.CDLL("/usr/local/cuda/lib64/libcudart.so.12")
        g_ms, n_g = timed(step_gather, args.steps, 2)
        tot = torch.tensor([n_tokens], dtype=torch.int64, device="cuda")
        dist.all_reduce(tot)
        if rank == 0:
            assert n_g == int(tot[0]), (n_g, int(tot[0]))
        gathered = {"value": BATCH * args.steps / (g_ms * 1e-3), "unit": "sentences/s", "ms_per_step": g_ms / args.steps,
                    "route": "device-resident shards; all_gather of token counts + NCCL send/recv of the 24-byte token "
                             "records to rank 0's GPU over NVLink (vibrato_b200.distributed.gather_token_records)",
                    "tokens_on_rank0": int(tot[0])}
        full = Inputs(utf8_all, off_all)
        torch.cuda.synchronize()
        wd_ms, _ = timed(lambda: step_device(full), args.steps, 2)
        we_ms, _ = timed(lambda: step_host(full), args.steps, 1)
        weak = {"value": BATCH * world * args.steps / (wd_ms * 1e-3), "unit": "sentences/s", "scaling": "weak",
                "batch_per_gpu": BATCH, "ms_per_step": wd_ms / args.steps,
                "e2e": {"value": BATCH * world * args.steps / (we_ms * 1e-3), "ms_per_step": we_ms / args.steps}}
    clocks = sampler.stop() if rank == 0 else None

    # per-rank figures that the line aggregates
    agg = torch.tensor([n_tokens, n_bytes, b_alg_viterbi, b_alg_step] + list(cnt), dtype=torch.float64, device="cuda")
    vit = torch.tensor([float(stage_acc[stage_names.index("viterbi")] / args.steps)], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(agg)
        dist.all_reduce(vit, op=dist.ReduceOp.MAX)
    tot_tokens, tot_bytes, b_alg_viterbi, b_alg_step = (float(x) for x in agg[:4])
    cnt = agg[4:].cpu().numpy()

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured copy bandwidth (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        st = stage_acc / args.steps
        vit_ms = float(vit[0])
        # the kernel of rank 0 processes its shard's share of the algorithmic bytes; all ranks run side by side
        achieved = (b_alg_viterbi / world) / (vit_ms * 1e-3) / 1e9
        traffic = traffic_src = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            if tj.get("dict") == cfg["dict"] and tj.get("batch") == BATCH and world == 1:
                traffic = tj.get("viterbi_dram_bytes_per_launch")
                traffic_src = tj.get("source")
        except Exception:
            pass
        # CPU baseline (rank 0, N=1 only): the oracle, one thread, bounded sample
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import vibrato_oracle as vo
            t = time.time()
            od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
            if user_csv is not None:
                od.set_user_csv(user_csv)
            n = min(cfg["cpu_sample"], BATCH)
            od.benchmark(utf8_all, off_all[: n // 10 + 1], n_threads=1, runs=1)  # warm-up (benchmark/src/main.rs:69-72)
            secs, _ = od.benchmark(utf8_all, off_all[: n + 1], n_threads=1, runs=2)
            cpu = {"value": 2 * n / secs, "unit": "sentences/s", "cores": 1, "kind": "port",
                   "sample": f"first {n} sentences of the batch x 2 runs, 1 thread; oracle = C restatement of vibrato "
                             "0.5.2 (Rust toolchain absent), body of benchmark/src/main.rs:53-65"}
            log(f"cpu baseline: {cpu['value']:.0f} sentences/s ({time.time() - t:.1f}s)")
        h2d = int(tot_bytes + (BATCH + world) * 8)
        d2h = int((BATCH + world) * 8 + tot_tokens * 24)
        line = {
            "metric": METRIC, "value": BATCH * args.steps / (dev_ms * 1e-3), "unit": "sentences/s", "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": workload_config(cfg_id, cfg),
            "e2e": {"value": BATCH * args.steps / (e2e_ms * 1e-3), "unit": "sentences/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps, "host_memory": "pinned",
                    "pageable": {"value": BATCH * args.steps / (e2e_pg_ms * 1e-3), "ms_per_step": e2e_pg_ms / args.steps,
                                 "host_memory": "pageable input (numpy arrays), staged through the library's pinned ring"},
                    "compact": {"value": BATCH * args.steps / (e2e_c_ms * 1e-3), "ms_per_step": e2e_c_ms / args.steps,
                                "d2h_bytes_per_step": int((BATCH + world) * 8 + tot_tokens * 16),
                                "what": "pinned buffers, tokenizer option compact_tokens: 16-byte records (byte range, "
                                        "word_idx, total_cost), character ranges rebuilt by the caller"}},
            "gpu_launches": int(launches_per_step * args.steps * world),
            "roofline": {"bound": "hbm", "kernel": "k_viterbi2", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": b_alg_viterbi / world, "kernel_ms": vit_ms,
                         "whole_step_algorithmic_bytes": b_alg_step,
                         "whole_step_achieved_GBs": b_alg_step / world / (dev_ms / args.steps * 1e-3) / 1e9},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "stage_ms": dict(zip(stage_names, [round(float(x), 4) for x in st])),
            "tokens_per_step": int(tot_tokens),
            "counters_per_sentence": dict(zip("U C M T P W E N K walks".split(), [round(float(x) / BATCH, 2) for x in cnt])),
        }
        if gathered:
            line["gathered"] = gathered
        if weak:
            line["weak"] = weak
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_tok_off, last_tokens, off)
        emit(line)
    lib().vbt_tokenizer_free(h)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("VBT_BENCH_CONFIG", "3")), choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the token offsets / records of the last timed step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if os.environ.get("VBT_BENCH_BATCH"):  # developer override (smoke runs)
        cfg["batch"] = int(os.environ["VBT_BENCH_BATCH"])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs writes the GPU arm's result on one GPU (--impl ours, --gpus 1)")
    if args.impl == "reference":
        run_reference(args, args.config, cfg, rank, world)
    else:
        run_ours(args, args.config, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
