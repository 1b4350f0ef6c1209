"""The n-gram LM fused into the CTC prefix beam search (velocity_asr.NGramLM, ctc_beam_search(lm_scorer=...)).

CPU: the oracle's ARPA back-off scorer against hand-computed values, the oracle search with lm_weight = 0, and the
loader's rejections (the C++ parser runs before any device call).  GPU: the scoring seam bit for bit against the
oracle, the fused search against the oracle's restatement of the rule, off-means-off, a known answer, errors."""
import ctypes
import math

import numpy as np
import pytest
import torch

import lm_oracle as LO
import velocity_oracle as O

HAND_ARPA = """\\data\\
ngram 1=7
ngram 2=4
ngram 3=2

\\1-grams:
-1.0\t<unk>
-99\t<s>\t-0.5
-0.5\ta\t-0.25
-0.75\tb\t-0.125
-1.25\tc\t0.25
-0.875\t<space>
-2.0\t</s>

\\2-grams:
-0.25\t<s> a\t-0.0625
-0.375\ta b\t0.125
-0.5\tb c
-0.625\ta <space>

\\3-grams:
-0.125\t<s> a b
-0.3\ta b c

\\end\\
"""


def vocab(V):
    import velocity_asr as va
    return va.create_default_vocabulary(max(V, 4))[:V]


def write(tmp_path, text, name="lm.arpa"):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def L(x):
    """an ARPA value as stored: log10 -> fp64 natural log -> fp32, back in fp64"""
    return float(np.float32(x * math.log(10)))


def f32(s):
    return float(np.float32(s))


# ------------------------------------------------------------------ CPU ------------------------------------
def test_oracle_scorer_hand_written_trigram(tmp_path):
    v = vocab(40)
    a, b, c, d, sp = (v.index(ch) for ch in "abcd ")
    lm = LO.ArpaLM.from_arpa(write(tmp_path, HAND_ARPA), v)
    assert lm.order == 3
    assert lm.lm((a,), b) == L(-0.125)                                   # listed trigram <s> a b
    assert lm.lm((c, a), c) == f32(L(-1.25) + L(-0.25) + 0.0)            # (c a) missing, (a) listed, unigram c
    assert lm.lm((a, b), d) == f32(L(-1.0) + L(-0.125) + L(0.125))       # <unk>, positive bow(a b)
    assert lm.lm((a,), sp) == f32(L(-0.625) + L(-0.0625))                # <space> is " ", bigram a <space>
    assert lm.lm((), a) == L(-0.25)                                      # short history starts at <s>
    assert lm.lm((), b) == f32(L(-0.75) + L(-0.5))                       # bow(<s>) then unigram b
    assert lm.lm((a, b), c) == L(-0.3)
    assert lm.lm((a, b), a) == f32(L(-0.5) + L(-0.125) + L(0.125))


def test_oracle_search_with_lm_weight_zero_is_lm_free(tmp_path):
    v = vocab(30)
    path = str(tmp_path / "r.arpa")
    LO.write_synthetic_arpa(path, v, order=3, seed=5)
    lm = LO.ArpaLM.from_arpa(path, v)
    lg = np.random.RandomState(3).standard_normal((2, 20, 30)).astype(np.float32) * 2
    assert LO.ctc_beam_search(lg, 5, lm_scorer=lm, lm_weight=0.0) == O.ctc_beam_search(lg, 5)
    assert LO.ctc_beam_search(lg, 5) == O.ctc_beam_search(lg, 5)
    assert LO.ctc_beam_search(lg, 5, lm_scorer=lm, lm_weight=1.0) != O.ctc_beam_search(lg, 5)


BAD = {
    "no_data": ("ngram 1=1\n\n\\1-grams:\n-1 a\n\\end\\\n", "line 6"),          # no \data\ anywhere
    "bad_count_line": ("\\data\\\nngram one=1\n", "line 2"),
    "count_mismatch": ("\\data\\\nngram 1=3\n\n\\1-grams:\n-1 <unk>\n-1 a\n\n\\end\\\n", "line 8"),
    "too_many": ("\\data\\\nngram 1=1\n\n\\1-grams:\n-1 <unk>\n-1 a\n\\end\\\n", "line 6"),
    "bad_number": ("\\data\\\nngram 1=2\n\n\\1-grams:\n-1 <unk>\n-1.x a\n\\end\\\n", "line 6"),
    "bad_bow": ("\\data\\\nngram 1=2\nngram 2=0\n\n\\1-grams:\n-1 <unk>\n-1 a nan\n\n\\2-grams:\n\n\\end\\\n",
                "line 7"),
    "no_end": ("\\data\\\nngram 1=1\n\n\\1-grams:\n-1 <unk>\n", "line 6"),
    "order_9": ("\\data\\\n" + "".join(f"ngram {n}=0\n" for n in range(1, 10)), "line 10"),
    "no_unk": ("\\data\\\nngram 1=1\n\n\\1-grams:\n-1 a\n\\end\\\n", "line 4"),
    "words": ("\\data\\\nngram 1=1\nngram 2=1\n\n\\1-grams:\n-1 <unk>\n\\2-grams:\n-1 a\n\\end\\\n", "line 8"),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_loader_rejects_malformed_arpa(tmp_path, case):
    import velocity_asr as va
    text, where = BAD[case]
    with pytest.raises(ValueError, match=where + ":"):
        va.NGramLM.from_arpa(write(tmp_path, text), vocab(10))


# ------------------------------------------------------------------ GPU ------------------------------------
@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


@pytest.mark.gpu
@pytest.mark.parametrize("order", [1, 2, 3, 4, 5])
def test_log_prob_seam_bit_exact(va, tmp_path, order):
    V = 60
    v = vocab(V)
    path = str(tmp_path / "r.arpa")
    LO.write_synthetic_arpa(path, v, order=order, seed=order, per_order=400)
    lm = va.NGramLM.from_arpa(path, v)
    ref = LO.ArpaLM.from_arpa(path, v)
    assert lm.order == order and lm.vocab_size == V
    rs = np.random.RandomState(order)
    grams = [g for g in ref.prob if len(g) > 1 and g[0] != "<s>"]
    prefixes = []
    for i in range(300):
        n = int(rs.randint(0, 12)) if i % 3 else int(rs.randint(0, 3))          # short and long
        p = [int(t) for t in rs.randint(1, V, size=n)]
        if grams and i % 2:                                                     # end on a listed context
            g = grams[rs.randint(len(grams))]
            p += [int(t) for t in g[:-1]]
        prefixes.append(p)
    toks = list(range(1, V))
    pre = [p for p in prefixes for _ in toks]
    tk = [t for _ in prefixes for t in toks]
    got = lm.log_prob(pre, tk).cpu().numpy()
    want = np.array([ref.lm(p, t) for p, t in zip(pre, tk)], np.float32)
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


# On the coarse-grid logits (golden1) two offers to one prefix from different alignments come within 1e-7 of each
# other at most weights: below the ulp noise between numpy's and the device's fp32 log-softmax tables, so which
# one wins (and hence the beam's last token) is the table's call, as in the LM-free search.  These weights keep
# every decision of that case at least 1e-3 apart in the oracle; the other cases are at least 4e-4 apart at 0.3 / 1.5.
GRID_WEIGHTS = {3: [0.5], 5: [0.3]}


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 5])
def test_beam_search_with_lm_matches_oracle(va, golden, tmp_path, order):
    for name, lg, W, blank in _search_cases(golden):
        V = lg.shape[-1]
        v = vocab(V)
        path = str(tmp_path / f"{name}.arpa")
        LO.write_synthetic_arpa(path, v, order=order, seed=order * 100 + V, blank_token=blank,
                                per_order=2000 if V >= 1000 else 200)
        lm = va.NGramLM.from_arpa(path, v, blank_token=blank)
        ref = LO.ArpaLM.from_arpa(path, v, blank_token=blank)
        weights = [0.7] if V >= 1000 else GRID_WEIGHTS[order] if name == "golden1" else [0.3, 1.5]
        for w in weights:
            res = va.ctc_beam_search(torch.from_numpy(lg).cuda(), beam_width=W, blank_token=blank,
                                     lm_weight=w, lm_scorer=lm)
            want = LO.ctc_beam_search(lg, W, blank_token=blank, lm_scorer=ref, lm_weight=w)
            for b, (beams, wb) in enumerate(zip(res, want)):
                assert [d.tokens for d in beams] == [t for t, _ in wb], (name, w, b)
                assert np.allclose([d.score for d in beams], [s for _, s in wb], rtol=0, atol=2e-4), (name, w, b)
        lm.close()


@pytest.mark.gpu
def test_lm_off_is_bit_identical(va, tmp_path):
    v = vocab(30)
    path = str(tmp_path / "r.arpa")
    LO.write_synthetic_arpa(path, v, order=3, seed=1)
    lm = va.NGramLM.from_arpa(path, v)
    lg = torch.from_numpy(np.random.RandomState(2).standard_normal((3, 40, 30)).astype(np.float32) * 2).cuda()
    plain = va.ctc_beam_search(lg, beam_width=6)
    for kw in ({"lm_scorer": lm, "lm_weight": 0.0}, {"lm_scorer": None, "lm_weight": 2.0}):
        other = va.ctc_beam_search(lg, beam_width=6, **kw)
        assert [[(d.tokens, d.score) for d in u] for u in other] == [[(d.tokens, d.score) for d in u] for u in plain]
    fused = va.ctc_beam_search(lg, beam_width=6, lm_scorer=lm, lm_weight=1.0)
    assert [[d.tokens for d in u] for u in fused] != [[d.tokens for d in u] for u in plain]


def _preference_arpa(tmp_path, good, bad, name):
    return write(tmp_path, "\\data\\\nngram 1=3\n\n\\1-grams:\n-3.0\t<unk>\n"
                           f"-0.1\t{good}\n-2.0\t{bad}\n\n\\end\\\n", name)


@pytest.mark.gpu
def test_lm_decides_between_acoustically_tied_tokens(va, tmp_path):
    v = vocab(12)
    a, b = v.index("a"), v.index("b")
    lg = np.full((1, 3, 12), -5.0, np.float32)
    lg[0, 0, a] = lg[0, 0, b] = 3.0                      # a and b tie; blanks after
    lg[0, 1:, 0] = 3.0
    lg = torch.from_numpy(lg).cuda()
    assert va.ctc_beam_search(lg, beam_width=4)[0][0].tokens == [a]          # the tie goes to the lower id
    prefer_b = va.NGramLM.from_arpa(_preference_arpa(tmp_path, "b", "a", "b.arpa"), v)
    prefer_a = va.NGramLM.from_arpa(_preference_arpa(tmp_path, "a", "b", "a.arpa"), v)
    assert va.ctc_beam_search(lg, beam_width=4, lm_scorer=prefer_b, lm_weight=0.5)[0][0].tokens == [b]
    assert va.ctc_beam_search(lg, beam_width=4, lm_scorer=prefer_a, lm_weight=0.5)[0][0].tokens == [a]
    dec = va.CTCDecoder(v)
    assert dec.decode_beam_search(lg, beam_width=4, lm_scorer=prefer_b, lm_weight=0.5) == ["b"]
    assert dec.decode_beam_search(lg, beam_width=4, lm_scorer=prefer_a, lm_weight=0.5) == ["a"]
    allb = dec.decode_beam_search(lg, beam_width=4, return_all_beams=True, lm_scorer=prefer_b, lm_weight=0.5)
    assert allb[0][0].text == "b" and allb[0][0].tokens == [b]


@pytest.mark.gpu
def test_lm_search_errors(va, tmp_path):
    from velocity_asr import _native
    v = vocab(20)
    path = str(tmp_path / "r.arpa")
    LO.write_synthetic_arpa(path, v, order=2, seed=3)
    lm = va.NGramLM.from_arpa(path, v)
    lg = torch.randn(1, 5, 20, device=lm.device)
    with pytest.raises(ValueError, match="vocabulary of 20"):
        va.ctc_beam_search(torch.randn(1, 5, 21, device=lm.device), lm_scorer=lm, lm_weight=1.0)
    with pytest.raises(ValueError, match="blank"):
        va.ctc_beam_search(lg, blank_token=3, lm_scorer=lm, lm_weight=1.0)
    # logits that are not on the LM's device are refused by the library before any launch
    host = np.zeros((1, 5, 20), np.float32)
    out_t = torch.empty(1, 2, 5, dtype=torch.int32, device=lm.device)
    out_l = torch.empty(1, 2, dtype=torch.int32, device=lm.device)
    out_s = torch.empty(1, 2, dtype=torch.float64, device=lm.device)
    with pytest.raises(ValueError, match="LM's device"):
        _native.check(_native.lib().vasr_ctc_beam_search_lm(
            host.ctypes.data_as(ctypes.c_void_p), 1, 5, 20, 2, 0, lm._handle, 1.0, _native.ptr(out_t),
            _native.ptr(out_l), _native.ptr(out_s), None))
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="the LM is on"):
            va.ctc_beam_search(lg.to("cuda:1"), lm_scorer=lm, lm_weight=1.0)
    with pytest.raises(NotImplementedError):
        va.ctc_beam_search(lg, lm_scorer=lambda prefix, tok: 0.0, lm_weight=1.0)
    lm.close()
    with pytest.raises(RuntimeError, match="closed"):
        va.ctc_beam_search(lg, lm_scorer=lm, lm_weight=1.0)
