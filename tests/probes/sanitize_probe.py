#!/usr/bin/env python3
"""Small end-to-end run for compute-sanitizer (memcheck / racecheck / initcheck), checked against the oracle;
lives under tests/ because only tests may use oracle/.   compute-sanitizer python tests/probes/sanitize_probe.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import vibrato_b200 as vb  # noqa: E402
from vibrato_b200 import synth  # noqa: E402
from oracle import vibrato_oracle as vo  # noqa: E402

g = json.load(open(os.path.join(ROOT, "tests", "golden", "vibrato_fixture.json"), encoding="utf-8"))
r = g["resources"]
d = vb.SystemDictionaryBuilder.from_readers(r["lex.csv"], r["matrix.def"], r["char.def"], r["unk.def"])
d.reset_user_lexicon_from_reader(r["user.csv"])
sents = [c["input"] for c in g["tokenizer_cases"]] * 20 + ["X" * 300, "", "0123456789" * 40]
for ign in (0, 1):
    tok = vb.Tokenizer.new(d).ignore_space(bool(ign)).max_grouping_len(24 if ign else 0)
    for chunk in (0, 100, 64):
        tok.set_option("chunk_sentences", chunk)
        res = tok.tokenize_batch(sents)
        print("ignore_space", ign, "chunk", chunk, "tokens", res.n_tokens, flush=True)
# every K3 instantiation the matrix connector can take (0 = 64-bit-address lookup, 1 = pruned, and its unpruned twin
# for a batch with a sentence of more than kPruneMaxChars characters)
for kernel, extra in ((0, []), (1, []), (1, ["X" * 16001])):
    tok = vb.Tokenizer.new(d).ignore_space(True)
    tok.set_option("viterbi_kernel", kernel)
    res = tok.tokenize_batch(sents + extra)
    print("viterbi_kernel", kernel, "long sentence", bool(extra), "tokens", res.n_tokens, flush=True)
sd = synth.make_dictionary("synth-tiny")
d2 = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
utf8, off = synth.make_corpus(sd, 2000, seed=9, log_uniform=(1, 200), unk_frac=0.1)
tok = vb.Tokenizer.new(d2)
tok.set_counting(True)
res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
tok_off, toks, cnt = od.tokenize_batch(utf8, off, want_counters=True)
assert res.tokens.tobytes() == toks.tobytes() and (tok.last_counters() == cnt).all()
print("synthetic ok", res.n_tokens)
# output stage (k_format_len / k_format_write), connection-id counters, Raw and Dual connector cost functions
for mode in ("mecab", "wakati", "detail"):
    tok.output_mode(mode)
    res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
    toff, text = res.text()
    eoff, etext = vo.format_batch(od, utf8, off, tok_off, toks, mode)
    assert text == etext and (toff == eoff).all(), mode
    print("output stage", mode, len(text), flush=True)
tok.output_mode(None)
tok.init_connid_counter()
tok.tokenize_batch(utf8=utf8, byte_offsets=off)
print("connid counts", [int(x.sum()) for x in tok.connid_counts()], flush=True)
right, left, cost = synth.make_bigram_files(sd, n_templates=12)
for dual in (False, True):
    dd = vb.SystemDictionaryBuilder.from_readers_with_bigram_info(sd.lex_csv, right, left, cost, sd.char_def, sd.unk_def,
                                                                   dual_connector=dual)
    odd = vo.OracleDictionary(sd.lex_csv, (right, left, cost), sd.char_def, sd.unk_def, dual_connector=dual)
    res = vb.Tokenizer.new(dd).tokenize_batch(utf8=utf8, byte_offsets=off)
    assert res.tokens.tobytes() == odd.tokenize_batch(utf8, off)[1].tobytes()
    print("bigram connector dual =", dual, res.n_tokens, flush=True)

# round 2: pool / character-estimate overflow retries, pageable input through the staging ring, the device-resident entry
# point, the multi-device engine on one device, a row longer than one staging pass (kPredCap) and a postings list beyond
# the segment buffer of k_candidates
tok = vb.Tokenizer.new(d2)
tok.set_option("pool_estimate_permille", 100)
tok.set_option("chars_estimate_permille", 20)
tok.set_option("chunk_sentences", 256)
res = tok.tokenize_batch(utf8=np.array(utf8, copy=True), byte_offsets=np.array(off, copy=True))
assert res.tokens.tobytes() == toks.tobytes()
print("retries + pageable ok", res.n_tokens, flush=True)
import torch  # noqa: E402
d_utf8 = torch.from_numpy(utf8).cuda()
d_off = torch.from_numpy(off.astype(np.int64)).cuda()
m = vb.Tokenizer.new(d2, devices=[0])
assert m.tokenize_batch_device(d_utf8.data_ptr(), d_off.data_ptr(), len(off) - 1, len(utf8))[2] == len(toks)
assert m.tokenize_batch(utf8=utf8, byte_offsets=off).tokens.tobytes() == toks.tobytes()
print("device-resident + multi engine ok", flush=True)
rows = "\n".join(f"a,1,1,{1000 - (i % 7)},h{i}" for i in range(600)) + "\nb,1,1,5,B\n"
dl = vb.SystemDictionaryBuilder.from_readers(rows, "2 2\n0 0 0\n0 1 0\n1 0 0\n1 1 0\n", "DEFAULT 0 1 0\n", "DEFAULT,0,0,30000,*\n")
ol = vo.OracleDictionary(rows, "2 2\n0 0 0\n0 1 0\n1 0 0\n1 1 0\n", "DEFAULT 0 1 0\n", "DEFAULT,0,0,30000,*\n")
for long in ([], ["b" * 16001]):  # pruned, then the unpruned twin
    u8, o = vb.Tokenizer.pack(["abab", "a", "bba"] * 5 + long)
    t = vb.Tokenizer.new(dl)
    assert t.tokenize_batch(utf8=u8, byte_offsets=o).tokens.tobytes() == ol.tokenize_batch(u8, o)[1].tobytes()
print("long rows ok", flush=True)
