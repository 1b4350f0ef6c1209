"""The word-level n-gram LM fused into the CTC prefix beam search (velocity_asr.WordNGramLM,
ctc_beam_search(lm_scorer=WordNGramLM, word_score=...)).

CPU: the oracle's word scorer against hand-computed values, the oracle search with the LM off, and the loader's
rejections (the C++ parser runs before any device call).  GPU: the scoring seam bit for bit against the oracle,
the fused search against the oracle's restatement of the rule (both modes), the lexicon constraint, known answers,
off-means-off and the error cases."""
import ctypes
import math
import string

import numpy as np
import pytest
import torch

import velocity_oracle as O
import word_lm_oracle as WO

HAND_ARPA = """\\data\\
ngram 1=6
ngram 2=3
ngram 3=1

\\1-grams:
-1.0\t<unk>
-99\t<s>\t-0.5
-0.5\tthe\t-0.25
-1.5\tcat\t-0.125
-1.25\tcot
-2.0\t</s>

\\2-grams:
-0.25\t<s> the\t-0.0625
-0.5\tthe cat\t0.125
-0.75\tcat </s>

\\3-grams:
-0.1\t<s> the cat

\\end\\
"""


def vocab(V):
    import velocity_asr as va
    return va.create_default_vocabulary(max(V, 4))[:V]


def word_vocab(V, blank):
    """For the golden shapes whose default vocabulary has no delimiter or fewer than three letters (V = 3, 5, 6):
    the delimiter and letters at non-blank ids, "<blank>" at the case's blank id."""
    base = (["<blank>", " "] + list(string.ascii_lowercase))[:V]
    return [base[(i - blank) % V] for i in range(V)]


def search_vocab(V, blank):
    return word_vocab(V, blank) if V < 9 else vocab(V)


def letters_of(v, blank):
    return [ch for i, ch in enumerate(v) if i != blank and ch in string.ascii_lowercase]


def write(tmp_path, text, name="w.arpa"):
    p = tmp_path / name
    p.write_text(text, encoding="utf-8")
    return str(p)


def L(x):
    return float(np.float32(x * math.log(10)))


def f32(s):
    return float(np.float32(s))


# ------------------------------------------------------------------ CPU ------------------------------------
def test_oracle_word_scorer_hand_written_trigram(tmp_path):
    lm = WO.WordLM(write(tmp_path, HAND_ARPA), vocab(40))
    assert lm.order == 3
    assert lm.words == ["<unk>", "the", "cat", "cot", "</s>"]
    assert sorted(lm.lexicon.values()) == [1, 2, 3]                            # <unk>, </s> are not in it
    assert lm.log_prob(["the"], "cat") == L(-0.1)                              # listed trigram <s> the cat
    assert lm.log_prob([], "the") == L(-0.25)
    assert lm.log_prob(["cat"], "</s>") == L(-0.75)                            # </s> is an ordinary word
    assert lm.log_prob(["the"], "cot") == f32(L(-1.25) + L(-0.25) + L(-0.0625))
    assert lm.log_prob(["dog"], "the") == f32(L(-0.5) + 0.0 + 0.0)             # dog is <unk>, no bow listed
    assert lm.log_prob(["the", "cat"], "zebra") == f32(L(-1.0) + L(-0.125) + L(0.125))


def test_oracle_split_and_spelling(tmp_path):
    v = vocab(40)
    lm = WO.WordLM(write(tmp_path, HAND_ARPA), v)
    t, h, e, c, a, o, sp, z = (v.index(ch) for ch in "thecao z")
    assert lm.split(()) == ((), ())
    assert lm.split((sp, t, h, e, sp, sp, c, a)) == ((1,), (c, a))           # empty runs close no word
    assert lm.split((z, sp, c, o, t, sp)) == ((0, 3), ())                     # unknown run -> <unk>
    assert (c, o) in lm.prefixes and (c, o, t) in lm.lexicon and (c, z) not in lm.prefixes


def test_oracle_search_with_lm_off_is_lm_free(tmp_path):
    v = vocab(30)
    path = str(tmp_path / "r.arpa")
    WO.write_synthetic_word_arpa(path, letters_of(v, 0), order=3, seed=5)
    lm = WO.WordLM(path, v)
    lg = np.random.RandomState(3).standard_normal((2, 20, 30)).astype(np.float32) * 2
    assert WO.ctc_beam_search(lg, 5, 0, lm, 0.0, 0.0) == O.ctc_beam_search(lg, 5)
    assert WO.ctc_beam_search(lg, 5, 0, lm, 1.0, 0.0) != O.ctc_beam_search(lg, 5)


BAD = {
    "count_mismatch": ("\\data\\\nngram 1=3\n\n\\1-grams:\n-1 <unk>\n-1 a\n\n\\end\\\n", "line 8"),
    "bad_number": ("\\data\\\nngram 1=2\n\n\\1-grams:\n-1 <unk>\n-1.x ab\n\\end\\\n", "line 6"),
    "no_end": ("\\data\\\nngram 1=1\n\n\\1-grams:\n-1 <unk>\n", "line 6"),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_word_loader_rejects_malformed_arpa(tmp_path, case):
    import velocity_asr as va
    text, where = BAD[case]
    with pytest.raises(ValueError, match=where + ":"):
        va.WordNGramLM.from_arpa(write(tmp_path, text), vocab(40))


def test_word_loader_rejections(tmp_path):
    import velocity_asr as va
    v = vocab(40)
    good = write(tmp_path, HAND_ARPA)
    with pytest.raises(ValueError, match="delimiter `|` is not in the vocabulary"):
        va.WordNGramLM.from_arpa(good, v, word_delimiter="|")
    with pytest.raises(ValueError, match="is the blank token"):
        va.WordNGramLM.from_arpa(good, v, blank_token=3)                       # v[3] == " "
    no_unk = write(tmp_path, "\\data\\\nngram 1=2\n\n\\1-grams:\n-1 cat\n-1 </s>\n\n\\end\\\n", "no_unk.arpa")
    with pytest.raises(ValueError, match="line 4: lexicon-free mode needs <unk>"):
        va.WordNGramLM.from_arpa(no_unk, v)
    unspellable = write(tmp_path, "\\data\\\nngram 1=3\n\n\\1-grams:\n-1 <unk>\n-1 #x\n-1 café\n\n\\end\\\n", "u.arpa")
    with pytest.raises(ValueError, match="lexicon-constrained mode needs a lexicon"):
        va.WordNGramLM.from_arpa(unspellable, v, lexicon_constrained=True)


# ------------------------------------------------------------------ GPU ------------------------------------
@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


@pytest.mark.gpu
@pytest.mark.parametrize("order", [1, 2, 3, 4, 5])
def test_word_log_prob_seam_bit_exact(va, tmp_path, order):
    v = vocab(40)
    path = str(tmp_path / "r.arpa")
    words = WO.write_synthetic_word_arpa(path, letters_of(v, 0), order=order, seed=order, n_words=60,
                                         per_order=400)
    lm = va.WordNGramLM.from_arpa(path, v)
    ref = WO.WordLM(path, v)
    assert lm.order == order and lm.lexicon_size == len(ref.lexicon) == len(words)
    rs = np.random.RandomState(order)
    pool = ref.words + ["<s>", "nosuchword", "café"]
    grams = [g for g in ref.arpa.prob if len(g) > 1 and g[0] != "<s>"]
    hists = []
    for i in range(300):
        h = [pool[j] for j in rs.randint(0, len(pool), size=int(rs.randint(0, 7)))]
        if grams and i % 2:                                                     # end on a listed context
            h += [ref.words[t] for t in grams[rs.randint(len(grams))][:-1]]
        hists.append(h)
    targets = ref.words + ["nosuchword"]
    hh = [h for h in hists for _ in targets]
    ww = [w for _ in hists for w in targets]
    got = lm.log_prob(hh, ww).cpu().numpy()
    want = np.array([ref.log_prob(h, w) for h, w in zip(hh, ww)], np.float32)
    assert np.array_equal(got.view(np.int32), want.view(np.int32)), np.abs(got - want).max()
    lm.close()


def _search_cases(golden):
    g = golden("beam")
    for i in range(int(g["n_cases"])):
        W, blank = (int(x) for x in g[f"par_{i}"])
        yield f"golden{i}", g[f"lg_{i}"], W, blank
    rs = np.random.RandomState(17)
    yield "W32", rs.standard_normal((2, 30, 40)).astype(np.float32) * 2.0, 32, 0
    yield "V1000", rs.standard_normal((2, 120, 1000)).astype(np.float32) * 3.0, 10, 0


# (lm_weight, word_score) pairs; one word_score is negative.  On the coarse-grid logits (golden1) offers from
# different alignments come within 6e-8 of each other at every weight: below the ulp noise between numpy's and the
# device's fp32 log-softmax tables, and moving single table entries by one ulp changes the oracle's own answer there
# at every pair tried.  Which alignment wins is the table's call, as in the LM-free search, so golden1 runs at pairs
# whose decisions come out the same on both tables in both modes at orders 3 and 5.
PAIRS = [(0.5, 1.0), (1.5, -0.75)]
GRID_PAIRS = [(0.5, 1.0), (0.5, -0.5)]


def _check(res, want, tag):
    for b, (beams, wb) in enumerate(zip(res, want)):
        assert [d.tokens for d in beams] == [t for t, _ in wb], (tag, b)
        assert np.allclose([d.score for d in beams], [s for _, s in wb], rtol=0, atol=2e-4), (tag, b)


@pytest.mark.gpu
@pytest.mark.parametrize("constrained", [False, True])
@pytest.mark.parametrize("order", [3, 5])
def test_word_beam_search_matches_oracle(va, golden, tmp_path, order, constrained):
    # The golden shapes at V < 9 are relabelled (word_vocab): golden1 (V = 6), golden2 (V = 3), golden6 (V = 5).
    for name, lg, W, blank in _search_cases(golden):
        V = lg.shape[-1]
        v = search_vocab(V, blank)
        path = str(tmp_path / f"{name}.arpa")
        WO.write_synthetic_word_arpa(path, letters_of(v, blank), order=order, seed=order * 100 + V,
                                     per_order=2000 if V >= 1000 else 200)
        lm = va.WordNGramLM.from_arpa(path, v, blank_token=blank, lexicon_constrained=constrained)
        ref = WO.WordLM(path, v, blank_token=blank, lexicon_constrained=constrained)
        pairs = PAIRS[:1] if V >= 1000 else GRID_PAIRS if name == "golden1" else PAIRS
        for w, ws in pairs:
            res = va.ctc_beam_search(torch.from_numpy(lg).cuda(), beam_width=W, blank_token=blank,
                                     lm_weight=w, lm_scorer=lm, word_score=ws)
            _check(res, WO.ctc_beam_search(lg, W, blank, ref, w, ws), (name, w, ws))
        lm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("constrained", [False, True])
def test_word_beam_search_on_spelled_words(va, tmp_path, constrained):
    v = vocab(40)
    path = str(tmp_path / "r.arpa")
    words = WO.write_synthetic_word_arpa(path, letters_of(v, 0), order=4, seed=9, n_words=50)
    lm = va.WordNGramLM.from_arpa(path, v, lexicon_constrained=constrained)
    ref = WO.WordLM(path, v, lexicon_constrained=constrained)
    rs = np.random.RandomState(4)
    lg = [WO.spelled_logits(v, [words[i] for i in rs.randint(0, len(words), size=6)], peak=8.0, noise=1.5, seed=s)
          for s in range(3)]
    n = min(x.shape[0] for x in lg)
    lg = np.stack([x[:n] for x in lg])
    for w, ws in PAIRS:
        res = va.ctc_beam_search(torch.from_numpy(lg).cuda(), beam_width=8, lm_weight=w, lm_scorer=lm, word_score=ws)
        want = WO.ctc_beam_search(lg, 8, 0, ref, w, ws)
        _check(res, want, (w, ws))
        assert any(v.index(" ") in d.tokens for u in res for d in u)           # words were closed
    lm.close()


@pytest.mark.gpu
def test_constrained_beams_spell_lexicon_words(va, tmp_path):
    v = vocab(30)
    path = str(tmp_path / "r.arpa")
    WO.write_synthetic_word_arpa(path, letters_of(v, 0), order=3, seed=2, n_words=30)
    lm = va.WordNGramLM.from_arpa(path, v, lexicon_constrained=True)
    ref = WO.WordLM(path, v, lexicon_constrained=True)
    lg = torch.from_numpy(np.random.RandomState(8).standard_normal((4, 40, 30)).astype(np.float32) * 2).cuda()
    for w in (0.0, 0.8):                                   # at lm_weight 0 the lexicon still constrains
        res = va.ctc_beam_search(lg, beam_width=6, lm_weight=w, lm_scorer=lm)
        for utt in res:
            assert 1 <= len(utt) <= 6
            for d in utt:
                _, u = ref.split(tuple(d.tokens))
                runs = "".join(v[t] for t in d.tokens).split(" ")
                assert all(tuple(v.index(ch) for ch in r) in ref.lexicon for r in runs if r), runs
                assert not u or u in ref.lexicon
    plain = va.ctc_beam_search(lg, beam_width=6)
    assert [[d.tokens for d in u] for u in res] != [[d.tokens for d in u] for u in plain]
    lm.close()


@pytest.mark.gpu
def test_word_lm_off_is_bit_identical(va, tmp_path):
    v = vocab(30)
    path = str(tmp_path / "r.arpa")
    WO.write_synthetic_word_arpa(path, letters_of(v, 0), order=3, seed=1)
    lm = va.WordNGramLM.from_arpa(path, v)
    lg = torch.from_numpy(np.random.RandomState(2).standard_normal((3, 40, 30)).astype(np.float32) * 2).cuda()
    plain = va.ctc_beam_search(lg, beam_width=6)
    off = va.ctc_beam_search(lg, beam_width=6, lm_scorer=lm, lm_weight=0.0, word_score=0.0)
    assert [[(d.tokens, d.score) for d in u] for u in off] == [[(d.tokens, d.score) for d in u] for u in plain]
    on = va.ctc_beam_search(lg, beam_width=6, lm_scorer=lm, lm_weight=1.0)
    assert [[d.tokens for d in u] for u in on] != [[d.tokens for d in u] for u in plain]
    lm.close()


def _cat_cot_arpa(tmp_path, good, bad):
    return write(tmp_path, "\\data\\\nngram 1=6\nngram 2=2\n\n\\1-grams:\n-3.0\t<unk>\n-99\t<s>\n-1.0\tthe\n"
                           f"-1.0\tcat\n-1.0\tcot\n-1.0\t</s>\n\n\\2-grams:\n-0.1\tthe {good}\n-2.0\tthe {bad}\n"
                           "\n\\end\\\n", f"{good}.arpa")


@pytest.mark.gpu
@pytest.mark.parametrize("constrained", [False, True])
def test_bigram_decides_acoustically_tied_words(va, tmp_path, constrained):
    v = vocab(40)
    lg = WO.spelled_logits(v, ["the", "cat"], noise=0.0)
    a, o = v.index("a"), v.index("o")
    rows = np.nonzero(lg[:, a] > 1.0)[0]
    lg[rows, o] = lg[rows, a]                               # "a" and "o" tie: cat / cot is acoustically even
    lg = torch.from_numpy(lg[None]).cuda()
    dec = va.CTCDecoder(v)
    for good, bad in (("cat", "cot"), ("cot", "cat")):
        lm = va.WordNGramLM.from_arpa(_cat_cot_arpa(tmp_path, good, bad), v, lexicon_constrained=constrained)
        assert dec.decode_beam_search(lg, beam_width=8, lm_scorer=lm, lm_weight=1.0) == [f"the {good}"]
        best = va.ctc_beam_search(lg, beam_width=8, lm_scorer=lm, lm_weight=1.0)[0][0]
        assert dec._tokens_to_text(best.tokens) == f"the {good}"
        lm.close()


@pytest.mark.gpu
def test_word_score_flips_split(va, tmp_path):
    v = vocab(40)
    a, b, sp = v.index("a"), v.index("b"), v.index(" ")
    lg = np.full((1, 4, 40), -5.0, np.float32)
    lg[0, 0, a] = 3.0
    lg[0, 1, 0] = lg[0, 1, sp] = 3.0                        # a blank or a space between "a" and "b": a tie
    lg[0, 2, b] = 3.0
    lg[0, 3, 0] = 3.0
    lg = torch.from_numpy(lg).cuda()
    path = write(tmp_path, "\\data\\\nngram 1=5\n\n\\1-grams:\n-1.0\t<unk>\n-1.0\ta\n-1.0\tb\n-1.0\tab\n-1.0\t</s>\n"
                           "\n\\end\\\n")
    lm = va.WordNGramLM.from_arpa(path, v)
    dec = va.CTCDecoder(v)
    assert dec.decode_beam_search(lg, beam_width=4, lm_scorer=lm, word_score=1.0) == ["a b"]
    assert dec.decode_beam_search(lg, beam_width=4, lm_scorer=lm, word_score=-1.0) == ["ab"]
    lm.close()


@pytest.mark.gpu
def test_word_lm_search_errors(va, tmp_path):
    from velocity_asr import _native
    v = vocab(20)
    path = str(tmp_path / "r.arpa")
    WO.write_synthetic_word_arpa(path, letters_of(v, 0), order=2, seed=3)
    lm = va.WordNGramLM.from_arpa(path, v)
    lg = torch.randn(1, 5, 20, device=lm.device)
    for kw in ({"lm_weight": -0.5}, {"lm_weight": math.inf}, {"lm_weight": math.nan},
               {"lm_weight": 1.0, "word_score": math.inf}, {"lm_weight": 1.0, "word_score": math.nan}):
        with pytest.raises(ValueError):
            va.ctc_beam_search(lg, lm_scorer=lm, **kw)
    with pytest.raises(ValueError, match="word_score needs a WordNGramLM"):
        va.ctc_beam_search(lg, word_score=1.0)
    tok_path = str(tmp_path / "t.arpa")
    import lm_oracle as LO
    LO.write_synthetic_arpa(tok_path, v, order=2, seed=3)
    tok_lm = va.NGramLM.from_arpa(tok_path, v)
    with pytest.raises(ValueError, match="word_score needs a WordNGramLM"):
        va.ctc_beam_search(lg, lm_scorer=tok_lm, lm_weight=1.0, word_score=1.0)
    with pytest.raises(ValueError, match="vocabulary of 20"):
        va.ctc_beam_search(torch.randn(1, 5, 21, device=lm.device), lm_scorer=lm, lm_weight=1.0)
    with pytest.raises(ValueError, match="blank"):
        va.ctc_beam_search(lg, blank_token=3, lm_scorer=lm, lm_weight=1.0)
    host = np.zeros((1, 5, 20), np.float32)
    out_t = torch.empty(1, 2, 5, dtype=torch.int32, device=lm.device)
    out_l = torch.empty(1, 2, dtype=torch.int32, device=lm.device)
    out_s = torch.empty(1, 2, dtype=torch.float64, device=lm.device)
    lib = _native.lib()
    with pytest.raises(ValueError, match="LM's device"):
        _native.check(lib.vasr_ctc_beam_search_word_lm(
            host.ctypes.data_as(ctypes.c_void_p), 1, 5, 20, 2, 0, lm._handle, 1.0, 0.0, _native.ptr(out_t),
            _native.ptr(out_l), _native.ptr(out_s), None))
    # each LM kind refuses the other's search at the C ABI
    with pytest.raises(ValueError, match="token LM"):
        _native.check(lib.vasr_ctc_beam_search_word_lm(
            _native.ptr(lg), 1, 5, 20, 2, 0, tok_lm._handle, 1.0, 0.0, _native.ptr(out_t), _native.ptr(out_l),
            _native.ptr(out_s), None))
    with pytest.raises(ValueError, match="word LM"):
        _native.check(lib.vasr_ctc_beam_search_lm(
            _native.ptr(lg), 1, 5, 20, 2, 0, lm._handle, 1.0, _native.ptr(out_t), _native.ptr(out_l),
            _native.ptr(out_s), None))
    with pytest.raises(ValueError, match="not a word LM"):
        _native.check(lib.vasr_lm_word_ids(tok_lm._handle, (ctypes.c_char_p * 1)(b"a"), 1,
                                           np.zeros(1, np.int32).ctypes.data_as(ctypes.c_void_p)))
    tok_lm.close()
    lm.close()
    with pytest.raises(RuntimeError, match="closed"):
        va.ctc_beam_search(lg, lm_scorer=lm, lm_weight=1.0)
    with pytest.raises(RuntimeError, match="closed"):
        lm.log_prob([[]], ["a"])
