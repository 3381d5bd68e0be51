#!/usr/bin/env python3
"""Developer tool: host-path (e2e) timing vs chunk size, with the per-stage sums of the chunked run."""
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
sd = synth.make_dictionary(name)
utf8, off = synth.make_corpus(sd, batch, seed=20260925)
d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
tok = vb.Tokenizer.new(d)
h_utf8 = torch.from_numpy(utf8).pin_memory().numpy()
h_off = torch.from_numpy(off.astype(np.int64)).pin_memory().numpy().view(np.uint64)
chunks = [int(x) for x in os.environ.get("VBT_PROBE_CHUNKS", "0,131072,262144,393216,524288").split(",")]
for chunk in chunks:
    tok.set_option("chunk_sentences", chunk)
    for _ in range(2):
        r = tok.tokenize_batch(utf8=h_utf8, byte_offsets=h_off)
        del r
    t = time.perf_counter()
    for _ in range(5):
        r = tok.tokenize_batch(utf8=h_utf8, byte_offsets=h_off)
        ms = tok.last_stage_ms()
        del r
    wall = (time.perf_counter() - t) / 5 * 1e3
    print(f"chunk={chunk:7d} e2e wall={wall:7.2f}ms  stage sum={sum(ms.values()):7.2f}  viterbi={ms['viterbi']:6.2f} "
          f"cand={ms['candidates']:5.2f} bt_write={ms['backtrack_write']:5.2f}", flush=True)
