#!/usr/bin/env python3
"""Developer tool: times the device-resident step for several k_viterbi2 lane layouts on one dictionary.
    python tools/sweep.py [dict] [batch] [fixed_len]"""
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import vibrato_b200 as vb  # noqa: E402
from vibrato_b200 import synth  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "synth-unidic"
batch = int(sys.argv[2]) if len(sys.argv) > 2 else 1000000
fixed = int(sys.argv[3]) if len(sys.argv) > 3 else 0
sd = synth.make_dictionary(name)
utf8, off = synth.make_corpus(sd, batch, seed=20260925, **({"fixed_len": fixed} if fixed else {}))
d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
tok = vb.Tokenizer.new(d)
d_utf8 = torch.from_numpy(utf8).cuda()
d_off = torch.from_numpy(off.astype(np.int64)).cuda()
torch.cuda.synchronize()
tag = os.environ.get("VBT_SWEEP_TAG", "")
for lanes, sort in [(8, 0), (16, 0)]:
    if True:
        tok.set_option("lanes_per_sentence", lanes)
        tok.set_option("sort_by_length", sort)
        for _ in range(2):
            tok.tokenize_batch_device(d_utf8.data_ptr(), d_off.data_ptr(), batch, len(utf8))
        acc = None
        t = time.perf_counter()
        for _ in range(3):
            tok.tokenize_batch_device(d_utf8.data_ptr(), d_off.data_ptr(), batch, len(utf8))
            ms = tok.last_stage_ms()
            acc = ms if acc is None else {k: acc[k] + v for k, v in ms.items()}
        wall = (time.perf_counter() - t) / 3 * 1e3
        print(f"{tag:14s} lanes={lanes:2d} sort={sort} wall={wall:7.2f}ms viterbi={acc['viterbi'] / 3:7.2f} "
              f"cand={acc['candidates'] / 3:6.2f} count={acc['count_chars'] / 3:5.2f} decode={acc['decode'] / 3:5.2f} scan_ends={acc['scan_ends'] / 3:5.2f} bt={(acc['backtrack_count'] + acc['backtrack_write']) / 3:5.2f} "
              f"sum={sum(acc.values()) / 3:7.2f}", flush=True)
