"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle (bit-exact) and
against the reference's golden vectors.  Run on the B200 box with `-m gpu`."""
import os

import numpy as np
import pytest

import vibrato_b200 as vb
from vibrato_b200 import synth
from oracle import vibrato_oracle as vo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dicts(golden, user=False):
    r = golden["resources"]
    d = vb.SystemDictionaryBuilder.from_readers(r["lex.csv"], r["matrix.def"], r["char.def"], r["unk.def"])
    od = vo.OracleDictionary(r["lex.csv"], r["matrix.def"], r["char.def"], r["unk.def"])
    if user:
        d.reset_user_lexicon_from_reader(r["user.csv"])
        od.set_user_csv(r["user.csv"])
    return d, od


def check_tokens(worker, exp_tokens):
    assert worker.num_tokens() == len(exp_tokens)
    for i, e in enumerate(exp_tokens):
        t = worker.token(i)
        assert t.surface() == e["surface"]
        assert [t.range_char().start, t.range_char().stop] == e["range_char"]
        assert [t.range_byte().start, t.range_byte().stop] == e["range_byte"]
        if "feature" in e:
            assert t.feature() == e["feature"]
        if "total_cost" in e:
            assert t.total_cost() == e["total_cost"]


def test_reference_golden_vectors(golden):
    # vibrato/src/tests/tokenizer.rs through Worker::reset_sentence / tokenize / token
    for case in golden["tokenizer_cases"]:
        d, _ = dicts(golden, case["user"])
        tok = vb.Tokenizer.new(d).ignore_space(case["ignore_space"]).max_grouping_len(case["max_grouping_len"])
        w = tok.new_worker()
        w.reset_sentence(case["input"])
        w.tokenize()
        if "tokens" in case:
            check_tokens(w, case["tokens"])
        else:
            assert w.num_tokens() == case["num_tokens"], case["name"]


def test_reference_repeat_and_iter(golden):
    d, _ = dicts(golden)
    w = vb.Tokenizer.new(d).new_worker()
    for text, n in golden["repeat_case"]["sequence"]:
        w.reset_sentence(text)
        w.tokenize()
        assert w.num_tokens() == n
        assert [t.surface() for t in w.token_iter()] == [w.token(i).surface() for i in range(n)]


def test_reference_mini_dictionaries(golden):
    for case in golden["mini_cases"]:
        d = vb.SystemDictionaryBuilder.from_readers(case["lex"], case["matrix"], case["char"], case["unk"])
        w = vb.Tokenizer.new(d).new_worker()
        w.reset_sentence(case["input"])
        w.tokenize()
        check_tokens(w, case["tokens"])


def test_detail_fields_match_oracle(golden):
    d, od = dicts(golden, True)
    tok = vb.Tokenizer.new(d)
    ow = od.worker()
    for text in ["京都東京都京都", "東京 都", "kampersandaX九"]:
        res = tok.tokenize_batch([text])
        exp = ow.tokenize(text)
        toks = res.sentence_tokens(0)
        assert len(toks) == len(exp)
        for t, e in zip(toks, exp):
            assert t.word_idx().packed == e["word_idx"] and t.feature() == e["feature"]
            assert (t.left_id(), t.right_id(), t.word_cost()) == od.word_param(e["word_idx"])


def assert_batch_equal(res, tok_off, toks):
    assert res.n_sent == len(tok_off) - 1
    np.testing.assert_array_equal(res.tok_offsets, tok_off)
    assert res.n_tokens == len(toks)
    for name in vb.TOKEN_DTYPE.names:
        np.testing.assert_array_equal(res.tokens[name], toks[name], err_msg=name)


@pytest.mark.parametrize("ignore_space,max_grouping", [(False, 0), (True, 0), (True, 24), (False, 3)])
def test_fixture_batch_matches_oracle(golden, ignore_space, max_grouping):
    d, od = dicts(golden, True)
    rng = np.random.default_rng(11)
    # the fixture unk.def covers DEFAULT / ALPHA / KANJI / KANJINUMERIC only: kana and NUMERIC characters
    # outside the lexicon dead-end the lattice (the reference panics there; we define "no tokens"),
    # so most sentences stay inside the covered classes and a minority exercises the dead end.
    covered = list("東京都大学院一二三九〇 xyzXabc京行") + ["  ", "𠮷", "é", "東京", "京都", "に", "た", "行く", "0", "7"]
    risky = covered + list("アイウ。、くっ")
    sents = ["".join(rng.choice(covered if i % 4 else risky, size=int(rng.integers(0, 40)))) for i in range(3000)]
    sents += [c["input"] for c in golden["tokenizer_cases"]] + ["", " ", "   ", "X" * 300, "0123456789" * 30]
    utf8, off = vb.Tokenizer.pack(sents)
    tok = vb.Tokenizer.new(d).ignore_space(ignore_space).max_grouping_len(max_grouping)
    tok.set_counting(True)
    res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
    tok_off, toks, cnt = od.tokenize_batch(utf8, off, ignore_space, max_grouping, n_threads=4, want_counters=True)
    assert_batch_equal(res, tok_off, toks)
    np.testing.assert_array_equal(tok.last_counters(), cnt)


@pytest.mark.parametrize("lanes,sort,chunk", [(4, 1, 0), (8, 0, 1000), (16, 1, 777), (32, 0, 0), (8, 1, 2500), (16, 0, 0),
                                              (32, 1, 1500)])
def test_viterbi_lane_layouts_match_oracle(lanes, sort, chunk):
    """Every lanes-per-sentence layout of k_viterbi, both sentence orders and the chunked (pipelined)
    host path give identical tokens."""
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 6001, seed=3, log_uniform=(1, 300), unk_frac=0.1, space_frac=0.02)
    # very long unknown words and rows with many nodes
    extra = ["abcdefghijklmnopqrstuvwxyzabcdefghijklmnopqrstuvwxyz" * 3 + "あいう", "12345678901234567890123456789012345あ",
             "あ" * 100, "ああああカタカナカタカナカタカナカタカナカタカナカタカナカタカナカタカナ漢字"]
    u2, o2 = vb.Tokenizer.pack(extra)
    utf8 = np.concatenate([utf8, u2])
    off = np.concatenate([off, o2[1:] + off[-1]])
    tok = vb.Tokenizer.new(d)
    tok.set_option("lanes_per_sentence", lanes)
    tok.set_option("sort_by_length", sort)
    tok.set_option("chunk_sentences", chunk)
    tok.set_option("dual_stream", lanes == 8)
    tok.set_counting(True)
    res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
    tok_off, toks, cnt = od.tokenize_batch(utf8, off, n_threads=8, want_counters=True)
    assert_batch_equal(res, tok_off, toks)
    np.testing.assert_array_equal(tok.last_counters(), cnt)
    res2 = tok.tokenize_batch(utf8=utf8, byte_offsets=off)  # again through the same tokenizer (buffers reused)
    assert_batch_equal(res2, tok_off, toks)


@pytest.mark.parametrize("user,ignore_space", [(False, False), (True, True)])
def test_synthetic_batch_matches_oracle(user, ignore_space):
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    ucsv = None
    if user:
        ucsv = synth.make_user_csv(sd, 500)
        d.reset_user_lexicon_from_reader(ucsv)
        od.set_user_csv(ucsv)
    utf8, off = synth.make_corpus(sd, 20000, log_uniform=(1, 256), unk_frac=0.15, space_frac=0.03, user_csv=ucsv,
                                  user_frac=0.05 if user else 0.0)
    tok = vb.Tokenizer.new(d).ignore_space(ignore_space).max_grouping_len(24 if ignore_space else 0)
    tok.set_counting(True)
    res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
    tok_off, toks, cnt = od.tokenize_batch(utf8, off, ignore_space, 24 if ignore_space else 0, n_threads=8,
                                           want_counters=True)
    assert_batch_equal(res, tok_off, toks)
    np.testing.assert_array_equal(tok.last_counters(), cnt)
    # a second, different batch through the same tokenizer (workspace reuse), counting off
    tok.set_counting(False)
    utf8b, offb = synth.make_corpus(sd, 5000, seed=77, fixed_len=512)
    resb = tok.tokenize_batch(utf8=utf8b, byte_offsets=offb)
    tok_offb, toksb, _ = od.tokenize_batch(utf8b, offb, ignore_space, 24 if ignore_space else 0, n_threads=8)
    assert_batch_equal(resb, tok_offb, toksb)


def test_edge_cases(golden):
    d, od = dicts(golden)
    tok = vb.Tokenizer.new(d)
    res = tok.tokenize_batch([])
    assert res.n_sent == 0 and res.n_tokens == 0
    res = tok.tokenize_batch(["", "", ""])
    assert list(res.tok_offsets) == [0, 0, 0, 0]
    for bad in (b"\xff", b"abc\xe3\x81", b"\xed\xa0\x80", b"\xc0\xaf"):
        with pytest.raises(vb.VibratoError) as ei:
            tok.tokenize_batch([b"ok", bad])
        assert ei.value.kind == "Utf8"
    # offsets that do not start at zero
    utf8, off = vb.Tokenizer.pack(["junk", "東京都", "京都"])
    res = tok.tokenize_batch(utf8=utf8, byte_offsets=off[1:])
    assert res.n_sent == 2 and [t.surface() for t in res.sentence_tokens(0)] == ["東京都"]
    # one very long sentence (deep lattice; > 32 predecessors and candidates per position via X homographs)
    long = ("X" * 50 + "東京都" + "9" * 70) * 40
    res = tok.tokenize_batch([long])
    tok_off, toks, _ = od.tokenize_batch(*vb.Tokenizer.pack([long]))
    assert_batch_equal(res, tok_off, toks)


def test_device_resident_api(golden):
    import torch
    d, od = dicts(golden, True)
    tok = vb.Tokenizer.new(d)
    sents = [c["input"] for c in golden["tokenizer_cases"]] * 50
    utf8, off = vb.Tokenizer.pack(sents)
    d_utf8 = torch.from_numpy(utf8.copy()).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    a, b, n = tok.tokenize_batch_device(d_utf8.data_ptr(), d_off.data_ptr(), len(sents), len(utf8))
    tok_off, toks, _ = od.tokenize_batch(utf8, off)
    assert n == len(toks)
    from cuda.bindings import runtime as cudart
    host = np.empty(n, dtype=vb.TOKEN_DTYPE)
    (err,) = cudart.cudaMemcpy(host.ctypes.data, b, n * 24, cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost)
    assert int(err) == 0
    host_off = np.empty(len(sents) + 1, dtype=np.uint64)
    (err,) = cudart.cudaMemcpy(host_off.ctypes.data, a, host_off.nbytes, cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost)
    assert int(err) == 0
    np.testing.assert_array_equal(host_off, tok_off)
    for name in vb.TOKEN_DTYPE.names:
        np.testing.assert_array_equal(host[name], toks[name])
    assert tok.last_launch_count() >= 7
    assert set(tok.last_stage_ms()) >= {"viterbi", "candidates"}


def test_blob_broadcast_path(golden):
    """Tokenizer built from a dictionary image that is already in device memory (the multi-GPU path)."""
    import ctypes as C
    import torch
    from vibrato_b200._native import check, lib
    d, od = dicts(golden)
    blob = torch.from_numpy(d.pack_blob()).cuda()
    h = C.c_void_p()
    check(lib().vbt_tokenizer_new_from_device_blob(blob.data_ptr(), blob.numel(), 0, 0, 0, C.byref(h)))
    try:
        utf8, off = vb.Tokenizer.pack(["京都東京都京都", "東京県に行く"])
        r = C.c_void_p()
        check(lib().vbt_tokenize_batch(h, utf8.ctypes.data, off.ctypes.data, 2, C.byref(r)))
        nt = C.c_uint64()
        check(lib().vbt_result_view(r, None, None, None, C.byref(nt)))
        assert nt.value == 3 + 4
        lib().vbt_result_free(r)
    finally:
        lib().vbt_tokenizer_free(h)


def test_cli_lookalikes(golden, tmp_path):
    """vibrato_b200/bin/{tokenize,benchmark}: the reference CLIs' flags and output formats
    (tokenize/src/main.rs:83-127, benchmark/src/main.rs:90-91)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "vibrato_b200", "bin", "tokenize")
    bexe = os.path.join(root, "vibrato_b200", "bin", "benchmark")
    if not os.path.exists(exe):
        pytest.skip("CLIs not built")
    for k, v in golden["resources"].items():
        (tmp_path / k).write_text(v, encoding="utf-8", newline="")
    _, od = dicts(golden, True)
    lines = ["京都東京都京都", "東京 都", "", "kampersanda", "東京県に行く"]
    text = ("\n".join(lines) + "\n").encode()
    ow = od.worker(ignore_space=True, max_grouping_len=24)
    exp = {"mecab": "", "wakati": "", "detail": ""}
    names = ["System", "User", "Unknown"]
    for ln in lines:
        toks = ow.tokenize(ln)
        exp["wakati"] += " ".join(t["surface"] for t in toks) + "\n"
        for t in toks:
            l, r, c = od.word_param(t["word_idx"])
            exp["mecab"] += f"{t['surface']}\t{t['feature']}\n"
            exp["detail"] += (f"{t['surface']}\t{t['feature']}\tlex_type={names[t['lex_type']]}\tleft_id={l}\t"
                              f"right_id={r}\tword_cost={c}\ttotal_cost={t['total_cost']}\n")
        exp["mecab"] += "EOS\n"
        exp["detail"] += "EOS\n"
    for mode in ("mecab", "wakati", "detail"):
        for where in ("device", "host"):  # text built by k_format_* on the GPU / by the C++ mirror of main.rs:83-127
            p = subprocess.run([exe, "-i", str(tmp_path), "-u", str(tmp_path / "user.csv"), "-O", mode, "-S", "-M", "24",
                                "--format-on", where], input=text, capture_output=True, timeout=120)
            assert p.returncode == 0, p.stderr.decode()
            assert p.stdout.decode() == exp[mode], (mode, where)
            assert p.stderr.decode().startswith("Loading the dictionary...\nReady to tokenize\n")
    p = subprocess.run([bexe, "-i", str(tmp_path)], input=text * 50, capture_output=True, timeout=300)
    assert p.returncode == 0, p.stderr.decode()
    out = p.stdout.decode().splitlines()
    assert out[0].startswith("Warmup: ") and out[1] == f"Number_of_sentences: {len(lines) * 50}"
    assert out[2].startswith("Elapsed_seconds_to_tokenize_all_sentences: [") and out[2].count(",") == 2


def test_one_very_long_sentence():
    """A 30 000-character sentence (MAX_SENTENCE_LENGTH is unbounded in the reference, common.rs:15)."""
    sd = synth.make_dictionary("synth-tiny")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 3, seed=4, fixed_len=30000, unk_frac=0.1)
    res = vb.Tokenizer.new(d).tokenize_batch(utf8=utf8, byte_offsets=off)
    tok_off, toks, _ = od.tokenize_batch(utf8, off)
    assert_batch_equal(res, tok_off, toks)


def test_many_prefix_hits_per_position():
    """More trie hits in one common-prefix walk than k_candidates' shared-memory hit buffer holds
    (keys a, aa, ..., a*14 in both lexicons), plus homograph lists longer than a warp."""
    lex = "".join(f"{'a' * k},{k % 3},{(k + 1) % 3},{100 * k},w{k}\n" for k in range(1, 15))
    lex += "".join(f"b,{i % 3},{(i * 7) % 3},{50 + i},h{i}\n" for i in range(70))
    matrix = "3 3\n" + "".join(f"{r} {l} {(r * 31 + l * 17) % 23 - 11}\n" for r in range(3) for l in range(3))
    chardef = "DEFAULT 0 1 0\nALPHA 1 1 0\n0x0061..0x007A ALPHA\n"
    unk = "DEFAULT,0,0,500,*\nALPHA,1,1,300,*\nALPHA,2,0,310,*\n"
    user = "".join(f"{'a' * k},{(k + 2) % 3},{k % 3},{90 * k},u{k}\n" for k in range(2, 12))
    d = vb.SystemDictionaryBuilder.from_readers(lex, matrix, chardef, unk).reset_user_lexicon_from_reader(user)
    od = vo.OracleDictionary(lex, matrix, chardef, unk).set_user_csv(user)
    sents = ["a" * 40, "b" * 5 + "a" * 20 + "b" * 3, "ab" * 30, "bbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbbb", "a" * 14 + "z" + "a" * 3]
    utf8, off = vb.Tokenizer.pack(sents * 40)
    for lanes in (8, 16, 32):
        tok = vb.Tokenizer.new(d)
        tok.set_option("lanes_per_sentence", lanes)
        tok.set_counting(True)
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        tok_off, toks, cnt = od.tokenize_batch(utf8, off, want_counters=True)
        assert_batch_equal(res, tok_off, toks)
        np.testing.assert_array_equal(tok.last_counters(), cnt)


def test_connid_counters_and_reordering(golden):
    """Worker::{init_connid_counter, update_connid_counts, compute_connid_probs} (worker.rs:77-103) on the
    device against the oracle, then the reference's reorder -> map flow (map/src/reorder.rs:24-66,
    map/src/main.rs:30-74): remapping connection ids must not change any token."""
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 4000, seed=21, log_uniform=(1, 120), unk_frac=0.1, space_frac=0.03)
    for ignore_space in (False, True):
        tok = vb.Tokenizer.new(d).ignore_space(ignore_space)
        tok.init_connid_counter()
        before = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        lid, rid = tok.connid_counts()
        olid, orid = od.connid_counts(utf8, off, ignore_space, n_threads=8)
        np.testing.assert_array_equal(lid, olid)
        np.testing.assert_array_equal(rid, orid)
        tok.tokenize_batch(utf8=utf8, byte_offsets=off)  # a second batch accumulates
        lid2, _ = tok.connid_counts()
        np.testing.assert_array_equal(lid2, 2 * olid)
    lprobs, rprobs = tok.compute_connid_probs()
    assert lprobs == vo.compute_connid_probs(2 * olid, 2 * orid)[0]
    d.map_connection_ids_from_iter([i for i, _ in lprobs], [i for i, _ in rprobs])
    tok2 = vb.Tokenizer.new(d).ignore_space(True)
    after = tok2.tokenize_batch(utf8=utf8, byte_offsets=off)
    assert_batch_equal(after, before.tok_offsets, before.tokens)
    # fixture: edges of one known lattice
    fd, fod = dicts(golden)
    t = vb.Tokenizer.new(fd)
    t.init_connid_counter()
    t.tokenize_batch(["京都東京都京都", "", "東京都"])
    u8, o = vb.Tokenizer.pack(["京都東京都京都", "", "東京都"])
    l1, r1 = t.connid_counts()
    l2, r2 = fod.connid_counts(u8, o)
    np.testing.assert_array_equal(l1, l2)
    np.testing.assert_array_equal(r1, r2)


def test_connid_counts_survive_a_pool_overflow_retry():
    """A batch whose candidate pool overflows is re-run from the start (engine.cu run_whole / run_host): the aborted
    attempt must not leave connection-id counts behind (lattice.rs:170-181 counts every lattice once)."""
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 3000, seed=33)
    olid, orid = od.connid_counts(utf8, off, False, n_threads=8)
    for chunk, what in ((0, "pool"), (512, "pool"), (0, "chars"), (512, "chars")):  # whole batch / chunked host pipeline
        tok = vb.Tokenizer.new(d)
        tok.set_option("chunk_sentences", chunk)
        tok.init_connid_counter()
        if what == "pool":
            tok.set_option("pool_estimate_permille", 100)  # far too small: the first attempt overflows
        else:  # the per-character launches are sized for fewer characters than the batch has: flagged, re-run
            tok.set_option("chars_estimate_permille", 20)
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        lid, rid = tok.connid_counts()
        np.testing.assert_array_equal(lid, olid)
        np.testing.assert_array_equal(rid, orid)
        otok_off, otoks, _ = od.tokenize_batch(utf8, off, n_threads=8)
        assert_batch_equal(res, otok_off, otoks)


def test_raw_connector_dictionary_matches_oracle():
    """Compact dictionary (RawConnector built from bigram.* files, builder.rs:111-148) on the device."""
    sd = synth.make_dictionary("synth-small")
    right, left, cost = synth.make_bigram_files(sd)
    d = vb.SystemDictionaryBuilder.from_readers_with_bigram_info(sd.lex_csv, right, left, cost, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, (right, left, cost), sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 5000, seed=8, log_uniform=(1, 200), unk_frac=0.1, space_frac=0.02)
    for lanes in (8, 16, 32):
        tok = vb.Tokenizer.new(d).ignore_space(True)
        tok.set_option("lanes_per_sentence", lanes)
        tok.set_counting(True)
        tok.init_connid_counter()
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        tok_off, toks, cnt = od.tokenize_batch(utf8, off, True, n_threads=8, want_counters=True)
        assert_batch_equal(res, tok_off, toks)
        np.testing.assert_array_equal(tok.last_counters(), cnt)
        lid, rid = tok.connid_counts()
        olid, orid = od.connid_counts(utf8, off, True, n_threads=8)
        np.testing.assert_array_equal(lid, olid)
        np.testing.assert_array_equal(rid, orid)
    d2 = vb.Dictionary.read(d.write())
    res2 = vb.Tokenizer.new(d2).ignore_space(True).tokenize_batch(utf8=utf8, byte_offsets=off)
    assert_batch_equal(res2, tok_off, toks)


def test_dual_connector_dictionary_matches_oracle():
    """Dual connector (dual_connector.rs; builder.rs:111-148 with dual_connector = true) on the device: the
    reduced-matrix gather plus the 8-lane scorer row give the oracle's lattice, counters and tokens, also after
    map_connection_ids and a trip through the .dic stream."""
    sd = synth.make_dictionary("synth-small")
    right, left, cost = synth.make_bigram_files(sd, n_templates=12)
    build = vb.SystemDictionaryBuilder.from_readers_with_bigram_info
    d = build(sd.lex_csv, right, left, cost, sd.char_def, sd.unk_def, dual_connector=True)
    od = vo.OracleDictionary(sd.lex_csv, (right, left, cost), sd.char_def, sd.unk_def, dual_connector=True)
    utf8, off = synth.make_corpus(sd, 5000, seed=9, log_uniform=(1, 200), unk_frac=0.1, space_frac=0.02)
    tok_off, toks, cnt = od.tokenize_batch(utf8, off, True, n_threads=8, want_counters=True)
    for lanes in (8, 16, 32):
        tok = vb.Tokenizer.new(d).ignore_space(True)
        tok.set_option("lanes_per_sentence", lanes)
        tok.set_counting(True)
        tok.init_connid_counter()
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        assert_batch_equal(res, tok_off, toks)
        np.testing.assert_array_equal(tok.last_counters(), cnt)
        lid, rid = tok.connid_counts()
        olid, orid = od.connid_counts(utf8, off, True, n_threads=8)
        np.testing.assert_array_equal(lid, olid)
        np.testing.assert_array_equal(rid, orid)
    # the Raw connector over the same files stores the same cost function
    raw = build(sd.lex_csv, right, left, cost, sd.char_def, sd.unk_def)
    assert_batch_equal(vb.Tokenizer.new(raw).ignore_space(True).tokenize_batch(utf8=utf8, byte_offsets=off), tok_off, toks)
    lmap = list(np.random.default_rng(3).permutation(np.arange(1, sd.num_left)))
    rmap = list(np.random.default_rng(4).permutation(np.arange(1, sd.num_right)))
    d.map_connection_ids_from_iter(lmap, rmap)
    d2 = vb.Dictionary.read(d.write())
    res2 = vb.Tokenizer.new(d2).ignore_space(True).tokenize_batch(utf8=utf8, byte_offsets=off)
    assert_batch_equal(res2, tok_off, toks)


def test_output_stage_matches_oracle_formatting(golden):
    """Device-side output stage (k_format_len / k_format_write) against the `tokenize` loop
    (tokenize/src/main.rs:83-127) applied to the oracle's tokens: all three modes, user + system + unknown
    words, empty sentences, sentences of more than 32 tokens, negative costs."""
    sd = synth.make_dictionary("synth-small")
    user = synth.make_user_csv(sd, 500)
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    d.reset_user_lexicon_from_reader(user)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od.set_user_csv(user)
    utf8, off = synth.make_corpus(sd, 3000, seed=21, log_uniform=(1, 300), unk_frac=0.15, space_frac=0.03,
                                  user_csv=user, user_frac=0.05)
    off = np.sort(np.concatenate([off, off[::50]])).astype(np.uint64)  # repeated offsets = empty sentences
    tok_off, toks = od.tokenize_batch(utf8, off, True, n_threads=8)[:2]
    assert int(np.diff(tok_off).max()) > 32 and int(np.diff(tok_off).min()) == 0
    tok = vb.Tokenizer.new(d).ignore_space(True)
    for mode in ("mecab", "wakati", "detail"):
        tok.output_mode(mode)
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        assert_batch_equal(res, tok_off, toks)
        toff, text = res.text()
        eoff, etext = vo.format_batch(od, utf8, off, tok_off, toks, mode)
        np.testing.assert_array_equal(toff, eoff)
        assert text == etext, mode
    tok.output_mode(None)
    res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
    with pytest.raises(vb.VibratoError):
        res.text()
    # golden dictionary: the exact lines of tests/tokenizer.rs rendered in mecab mode
    gd, god = dicts(golden, True)
    gt = vb.Tokenizer.new(gd).ignore_space(True).output_mode("detail")
    sents = ["京都東京都京都", "", "東京 都", "kampersanda"]
    u8, o = vb.Tokenizer.pack(sents)
    res = gt.tokenize_batch(utf8=u8, byte_offsets=o)
    eoff, etext = vo.format_batch(god, u8, o, *god.tokenize_batch(u8, o, True)[:2], "detail")
    toff, text = res.text()
    assert text == etext and list(toff) == list(eoff)


def _gold_corpus(od, sentences, rng, merge_frac=0.1, feat_frac=0.1):
    """`surface\\tfeature` / `EOS` corpus from the oracle's own analysis, with some tokens merged and some features
    altered so that precision and recall are not trivially 1."""
    w = od.worker(ignore_space=False)
    lines = []
    for s in sentences:
        toks = w.tokenize(s)
        i = 0
        while i < len(toks):
            t = toks[i]
            surface, feature = t["surface"], t["feature"]
            if i + 1 < len(toks) and rng.random() < merge_frac:
                surface += toks[i + 1]["surface"]
                i += 1
            elif rng.random() < feat_frac:
                feature = "X," + feature if rng.random() < 0.5 else feature + ",extra"  # first / a later field differs
            lines.append(f"{surface}\t{feature}")
            i += 1
        lines.append("EOS")
    return "\n".join(lines) + "\n"


def test_evaluate_matches_reference_loop(golden, tmp_path):
    """vbt_evaluate / bin/evaluate against the loop of evaluate/src/main.rs:61-138 restated over oracle tokens."""
    import os
    import subprocess
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 400, seed=33, log_uniform=(1, 120), unk_frac=0.1, space_frac=0.0)
    buf = bytes(memoryview(utf8))
    sents = [buf[int(off[i]):int(off[i + 1])].decode() for i in range(len(off) - 1)]
    rng = np.random.default_rng(5)
    tok = vb.Tokenizer.new(d)
    exact = _gold_corpus(od, sents, rng, 0.0, 0.0)
    r = tok.evaluate(exact)
    assert r["num_ref"] == r["num_sys"] == r["num_cor"] > 1000 and r["f1"] == 1.0
    corpus = _gold_corpus(od, sents, rng) + "\t\nEOS\nEOS\n"  # an example without input is dropped (corpus.rs:105-108)
    for idx in ((), (0,), (0, 1, 40)):
        r = tok.evaluate(corpus, idx)
        assert (r["num_ref"], r["num_sys"], r["num_cor"]) == vo.evaluate_corpus(od, corpus, idx)
        assert 0.5 < r["precision"] < 1.0 and 0.5 < r["recall"] < 1.0
    assert tok.evaluate(corpus, (0,))["num_cor"] > tok.evaluate(corpus)["num_cor"]
    for bad in ("a\tb\tc\nEOS\n", "abc\nEOS\n", "\nEOS\n"):  # corpus.rs:111-116
        with pytest.raises(vb.VibratoError) as ei:
            tok.evaluate(bad)
        assert ei.value.kind == "InvalidFormat"
    # max_grouping_len is the one tokenizer knob the tool exposes (main.rs:72)
    r24 = vb.Tokenizer.new(d).max_grouping_len(3).evaluate(corpus)
    assert (r24["num_ref"], r24["num_sys"], r24["num_cor"]) == vo.evaluate_corpus(od, corpus, (), 3)
    # the CLI: flags and the three output lines (main.rs:13-38, :132-136)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "vibrato_b200", "bin", "evaluate")
    if not os.path.exists(exe):
        pytest.skip("CLIs not built")
    for k, v in golden["resources"].items():
        (tmp_path / k).write_text(v, encoding="utf-8", newline="")
    gd, god = dicts(golden, True)
    gold = "京都\t京都,名詞,固有名詞,地名,一般,*,*,キョウト,京都,*,A,*,*,*,1/5\n東京都\tX\nEOS\n東京\tY\n都\tZ\nEOS\n"
    p = subprocess.run([exe, "-t", "/dev/stdin", "-i", str(tmp_path), "-u", str(tmp_path / "user.csv"), "--feature-indices", "0"],
                       input=gold.encode(), capture_output=True, timeout=120)
    assert p.returncode == 0, p.stderr.decode()
    nr, ns, nc = vo.evaluate_corpus(god, gold, (0,))
    pr, rc = nc / ns, nc / nr
    f1 = 2 * pr * rc / (pr + rc) if pr + rc else float("nan")
    fmt = lambda v: "NaN" if v != v else (repr(v)[:-2] if repr(v).endswith(".0") else repr(v))  # Rust `{}` for f64
    assert p.stdout.decode() == f"Precision = {fmt(pr)}\nRecall = {fmt(rc)}\nF1 = {fmt(f1)}\n"
    assert p.stderr.decode().startswith("Loading the dictionary...\nTokenizing...\n")


def test_output_stage_and_evaluate_edge_cases(golden):
    """Empty batch, only-empty sentences and an empty corpus through the output stage and the evaluate loop."""
    d, od = dicts(golden)
    tok = vb.Tokenizer.new(d)
    for mode, term in (("mecab", b"EOS\n"), ("wakati", b"\n"), ("detail", b"EOS\n")):
        tok.output_mode(mode)
        res = tok.tokenize_batch([])
        toff, text = res.text()
        assert res.n_sent == 0 and text == b"" and list(toff) == [0]
        res = tok.tokenize_batch(["", "", ""])
        toff, text = res.text()
        assert res.n_tokens == 0 and text == term * 3 and list(toff) == [len(term) * i for i in range(4)]
        res = tok.tokenize_batch(["", "京都", ""])
        toff, text = res.text()
        u8, o = vb.Tokenizer.pack(["", "京都", ""])
        eoff, etext = vo.format_batch(od, u8, o, *od.tokenize_batch(u8, o)[:2], mode)
        assert text == etext and list(toff) == list(eoff)
    tok.output_mode(None)
    for corpus in ("", "EOS\n", "EOS\nEOS\n", "京都\tX\n"):  # no example at all (a trailing sentence without EOS is dropped)
        r = tok.evaluate(corpus)
        assert (r["num_ref"], r["num_sys"], r["num_cor"]) == (0, 0, 0) and r["precision"] != r["precision"]
    with pytest.raises(vb.VibratoError) as ei:
        tok.evaluate(b"\xff\tX\nEOS\n")
    assert ei.value.kind == "StdIo"


def test_malformed_byte_offsets_are_refused(golden):
    """The C ABI takes offsets instead of strings: decreasing offsets are a caller error that must come back as
    InvalidArgument (vbt_tokenize_batch checks its host array; device-resident offsets are checked by k_count_chars,
    after which every later kernel of the batch stands down), and the tokenizer must stay usable."""
    d, od = dicts(golden)
    tok = vb.Tokenizer.new(d)
    u8, o = vb.Tokenizer.pack(["京都東京都京都", "東京都", "京都"])
    good = tok.tokenize_batch(utf8=u8, byte_offsets=o)
    bad = o.copy()
    bad[1], bad[2] = o[2], o[1]  # 0, 30, 21, 36: sentence 1 runs backwards, sentence 2 overlaps sentence 0
    for chunk in (0, 1):
        tok.set_option("chunk_sentences", chunk)
        with pytest.raises(vb.VibratoError) as ei:
            tok.tokenize_batch(utf8=u8, byte_offsets=bad)
        assert ei.value.kind == "InvalidArgument"
        again = tok.tokenize_batch(utf8=u8, byte_offsets=o)
        assert again.tokens.tobytes() == good.tokens.tobytes()


def test_validation_kit_runs_end_to_end(golden, tmp_path):
    """tools/validate_dic.py (the check for the day a released dictionary is mounted) on a zstd-compressed `.dic`
    written from the fixture sources: load, audit, rewrite and the GPU tokenisation step all run; the README
    comparison itself needs the real ipadic and is reported as plain output here."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import validate_dic
    d, _ = dicts(golden)
    path = tmp_path / "system.dic.zst"
    path.write_bytes(validate_dic.zstd_compress(d.write()))
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "validate_dic.py"), str(path)], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "[PASS] write(read(x)) == x" in p.stdout and "[PASS] audit system lexicon" in p.stdout
    assert "--- `mens second bag` -O mecab -S -M 24" in p.stdout


def test_device_resident_offsets_are_checked_on_the_device(golden):
    """vbt_tokenize_batch_device cannot look at its offsets on the host: k_count_chars flags decreasing or
    out-of-buffer values, every later kernel of the batch stands down, and the call fails with InvalidArgument."""
    import torch
    d, _ = dicts(golden)
    tok = vb.Tokenizer.new(d)
    u8, off = vb.Tokenizer.pack(["東京都に行く", "京都", "大阪"])
    d_utf8 = torch.from_numpy(u8.copy()).cuda()
    good = tok.tokenize_batch_device(d_utf8.data_ptr(), torch.from_numpy(off.astype(np.int64)).cuda().data_ptr(), 3, len(u8))
    assert good[2] > 0
    for bad in ([0, 18, 12, 30], [0, 18, 24, 31], [5, 3, 24, 30]):  # decreasing; past the buffer; decreasing at the start
        o = torch.tensor(bad, dtype=torch.int64).cuda()
        with pytest.raises(vb.VibratoError) as ei:
            tok.tokenize_batch_device(d_utf8.data_ptr(), o.data_ptr(), 3, len(u8))
        assert ei.value.kind == "InvalidArgument"
    # the tokenizer is still usable afterwards
    again = tok.tokenize_batch_device(d_utf8.data_ptr(), torch.from_numpy(off.astype(np.int64)).cuda().data_ptr(), 3, len(u8))
    assert again[2] == good[2]


def test_compact_token_records_match_the_full_ones():
    """Tokenizer option compact_tokens: 16-byte records (vbt_token16) from the device, expanded on the host, equal the
    24-byte records and the oracle — whole batch, chunked host pipeline, small-batch path, multi-device engine and
    the device-resident entry point; the two result views refuse each other's results."""
    import torch
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 3000, seed=12, log_uniform=(1, 150), unk_frac=0.1, space_frac=0.03, astral_frac=0.01)
    otok_off, otoks, _ = od.tokenize_batch(utf8, off, ignore_space=True, n_threads=8)
    for devices, chunk in ((None, 0), (None, 512), ([0], 0)):
        tok = vb.Tokenizer.new(d, devices=devices).ignore_space(True).compact_tokens(True)
        tok.set_option("chunk_sentences", chunk)
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        assert res.compact is not None and res.compact.dtype.itemsize == 16
        assert_batch_equal(res, otok_off, otoks)
    small = tok.tokenize_batch(["東京都に行く", "", "abc def"])  # the single-synchronisation path
    full = vb.Tokenizer.new(d).ignore_space(True).tokenize_batch(["東京都に行く", "", "abc def"])
    assert_batch_equal(small, full.tok_offsets, full.tokens)
    # device-resident: d_tokens are vbt_token16 records
    d_utf8 = torch.from_numpy(utf8).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    one = vb.Tokenizer.new(d).ignore_space(True).compact_tokens(True)
    p_off, p_tok, n_tok = one.tokenize_batch_device(d_utf8.data_ptr(), d_off.data_ptr(), len(off) - 1, len(utf8))
    got = _device_bytes(p_tok, n_tok * 16).view(vb.COMPACT_TOKEN_DTYPE)
    for name in vb.COMPACT_TOKEN_DTYPE.names:
        np.testing.assert_array_equal(got[name], otoks[name], err_msg=name)
    # the views do not mix, and the output stage needs full records
    import ctypes as C
    from vibrato_b200._native import lib
    r = C.c_void_p()
    u8, o = vb.Tokenizer.pack(["東京都"])
    assert lib().vbt_tokenize_batch(one.handle(), u8.ctypes.data, o.ctypes.data, 1, C.byref(r)) == 0
    pt = C.c_void_p()
    assert lib().vbt_result_view(r, None, C.byref(pt), None, None) != 0
    assert lib().vbt_result_view_compact(r, None, C.byref(pt), None, None) == 0
    lib().vbt_result_free(r)
    with pytest.raises(vb.VibratoError):
        one.output_mode("mecab")


def _device_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.parametrize("n_dev", [1, 2, 4, 8])
def test_multi_device_tokenizer_matches_single_device(n_dev):
    """vbt_tokenizer_new_multi (SURVEY.md 8(e)): shards by bytes, one result in input order, byte-identical to the
    single-device tokenizer and to the oracle; the device-resident route gathers the same records on devices[0].
    n_dev = 1 runs the multi-device code path on one GPU; larger counts need that many GPUs and skip otherwise."""
    import torch
    if _device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    sd = synth.make_dictionary("synth-small")
    d = vb.SystemDictionaryBuilder.from_readers(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    od = vo.OracleDictionary(sd.lex_csv, sd.matrix, sd.char_def, sd.unk_def)
    utf8, off = synth.make_corpus(sd, 5000, seed=77, log_uniform=(1, 200), unk_frac=0.1, space_frac=0.02)
    single = vb.Tokenizer.new(d).ignore_space(True)
    multi = vb.Tokenizer.new(d, devices=list(range(n_dev))).ignore_space(True)
    info = multi.describe()
    assert info["devices"] == list(range(n_dev))
    if n_dev > 1:
        assert info["dictionary_transport"].startswith("nccl") or info["dictionary_transport"] == "cudaMemcpyPeer"
    otok_off, otoks, _ = od.tokenize_batch(utf8, off, ignore_space=True, n_threads=8)
    ref = single.tokenize_batch(utf8=utf8, byte_offsets=off)
    assert_batch_equal(ref, otok_off, otoks)
    for _ in range(2):  # the second call reuses workspaces and the pinned result pool
        res = multi.tokenize_batch(utf8=utf8, byte_offsets=off)
        assert_batch_equal(res, otok_off, otoks)
    # edge cases: fewer sentences than devices, empty sentences, empty batch
    for sents in (["東京都"], ["", "", ""], [], ["a"] * 3 + [""] * 5):
        u8, o = vb.Tokenizer.pack(sents)
        a = single.tokenize_batch(utf8=u8, byte_offsets=o)
        b = multi.tokenize_batch(utf8=u8, byte_offsets=o)
        assert_batch_equal(b, a.tok_offsets, a.tokens)
    # device-resident input on devices[0]; results gathered there
    torch.cuda.set_device(0)
    d_utf8 = torch.from_numpy(utf8).cuda()
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    p_off, p_tok, n_tok = multi.tokenize_batch_device(d_utf8.data_ptr(), d_off.data_ptr(), len(off) - 1, len(utf8))
    assert n_tok == len(otoks)
    got_off = _device_bytes(p_off, (len(off)) * 8).view("<u8")
    got_tok = _device_bytes(p_tok, n_tok * 24).view(vb.TOKEN_DTYPE)
    np.testing.assert_array_equal(got_off, otok_off)
    for name in vb.TOKEN_DTYPE.names:
        np.testing.assert_array_equal(got_tok[name], otoks[name], err_msg=name)
    # connection-id counters add up over the devices
    multi2 = vb.Tokenizer.new(d, devices=list(range(n_dev)))
    multi2.init_connid_counter()
    multi2.tokenize_batch(utf8=utf8, byte_offsets=off)
    lid, rid = multi2.connid_counts()
    olid, orid = od.connid_counts(utf8, off, False, n_threads=8)
    np.testing.assert_array_equal(lid, olid)
    np.testing.assert_array_equal(rid, orid)


def _device_bytes(ptr, nbytes):
    """Device memory -> numpy bytes through the CUDA runtime (cudaMemcpyDefault: the address says where it lives)."""
    from cuda.bindings import runtime as cudart
    host = np.empty(max(nbytes, 1), dtype=np.uint8)
    (err,) = cudart.cudaMemcpy(host.ctypes.data, ptr, nbytes, cudart.cudaMemcpyKind.cudaMemcpyDefault)
    assert int(err) == 0, err
    return host[:nbytes]


def test_row_longer_than_u16_follows_the_reference_truncation():
    """lattice.rs:144 stores the best predecessor's row index as u16.  With more than 65 536 nodes in one `ends` row
    the index wraps and the backtrack follows a different node than the one that gave the minimum — what the
    reference does is the specification, and the oracle restates it.  70 000 homographs of one surface also drive
    k_candidates' per-thread fallback (a postings list beyond the segment buffer's 255) and k_viterbi2's multi-pass
    staging (rows longer than kPredCap)."""
    n = 70000
    best = 69000  # the cheapest homograph sits beyond u16: 69000 as u16 = 3464
    rows = [f"a,1,1,{1000 if i != best else 10},h{i}" for i in range(n)] + ["b,1,1,5,B"]
    lex = "\n".join(rows) + "\n"
    matrix = "2 2\n0 0 0\n0 1 0\n1 0 0\n1 1 0\n"
    char_def, unk_def = "DEFAULT 0 1 0\n", "DEFAULT,0,0,30000,*\n"
    d = vb.SystemDictionaryBuilder.from_readers(lex, matrix, char_def, unk_def)
    od = vo.OracleDictionary(lex, matrix, char_def, unk_def)
    utf8, off = vb.Tokenizer.pack(["ab", "a", "ba", "abab"])
    otok_off, otoks, _ = od.tokenize_batch(utf8, off)
    for kernel in (1, 2, 0):
        tok = vb.Tokenizer.new(d)
        tok.set_option("viterbi_kernel", kernel)
        res = tok.tokenize_batch(utf8=utf8, byte_offsets=off)
        assert_batch_equal(res, otok_off, otoks)
    first = res.sentence_tokens(0)[0]
    assert first.feature() == f"h{best & 0xFFFF}"  # the truncated index, as in the reference
    assert res.sentence_tokens(1)[0].feature() == f"h{best & 0xFFFF}"  # insert_eos goes through the same u16 (lattice.rs:85-101)
