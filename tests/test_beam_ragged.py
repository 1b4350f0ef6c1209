"""Ragged batches in the device CTC prefix beam search, and the fused PCM -> n-best path.

ctc_beam_search(logits, lengths=...) searches utterance b over its first lengths[b] frames only
(vasr_ctc_beam_search_ragged); VELOCITYASR.transcribe_beam(pcm, lengths=...) runs log-mel, forward and the search in
one native call (vasr_transcribe_beam / _host).  Both promise bit-for-bit equality, fp64 scores included, with the
same search run on each utterance alone, so the comparisons below use == and no tolerance.

CPU: malformed lengths are refused before any device work, in Python and at the C ABI.  GPU: ragged equals alone
for every search kind, widths and vocabularies; one ragged case against the oracles; fused equals composed in both
scan modes, through device and pinned host PCM, for the fp32 and the FakeQuantize model; the error cases."""
import ctypes
import string

import numpy as np
import pytest
import torch

import fixtures_util as FU
import lm_oracle as LO
import velocity_oracle as O
import word_lm_oracle as WO

KINDS = ["none", "token3", "token5", "word", "word_constrained"]
TOKEN_WEIGHT = 0.7
WORD_WEIGHT, WORD_SCORE = 0.5, 1.0


def vocab(V):
    import velocity_asr as va
    return va.create_default_vocabulary(max(V, 4))[:V]


def letters_of(v):
    return [ch for i, ch in enumerate(v) if i != 0 and ch in string.ascii_lowercase]


def beams_of(res):
    """Everything a result carries, for exact comparison: per utterance [(tokens, fp64 score), ...]."""
    return [[(d.tokens, d.score) for d in utt] for utt in res]


# ------------------------------------------------------------------ CPU ------------------------------------
def test_malformed_lengths_raise_before_device_work():
    import velocity_asr as va
    lg = torch.zeros(3, 5, 4)                       # host logits: a device call would come after the checks
    with pytest.raises(RuntimeError, match="expected 3 lengths"):
        va.ctc_beam_search(lg, lengths=[1, 2])
    with pytest.raises(RuntimeError, match=r"in \[0, 5\]"):
        va.ctc_beam_search(lg, lengths=[1, -1, 2])
    with pytest.raises(RuntimeError, match=r"in \[0, 5\]"):
        va.ctc_beam_search(lg, lengths=torch.tensor([6, 1, 2]))
    with pytest.raises(RuntimeError, match="expected 3 lengths"):
        va.CTCDecoder(vocab(4)).decode_beam_search(lg, lengths=(1, 2, 3, 4))


@pytest.mark.parametrize("bad", [[-1, 2], [2, 6]])
def test_c_abi_checks_row_lengths_first(bad):
    """vasr_ctc_beam_search_ragged refuses a length outside [0, L] with VASR_ERR_SHAPE before touching a device."""
    from velocity_asr import _native
    host = np.zeros((2, 5, 4), np.float32)
    rows = np.asarray(bad, np.int32)
    out = np.zeros(64, np.int32)
    scores = np.zeros(4, np.float64)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    with pytest.raises(RuntimeError, match="between 0 and L frames"):
        _native.check(_native.lib().vasr_ctc_beam_search_ragged(p(host), p(rows), 2, 5, 4, 2, 0, None, 0.0, 0.0,
                                                                p(out), p(out), p(scores), None))


# ------------------------------------------------------------------ GPU ------------------------------------
@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


def make_lm(va, kind, v, tmp_path, seed=0):
    """(device LM, oracle LM, search kwargs) for one search kind over vocabulary v."""
    if kind == "none":
        return None, None, {}
    path = str(tmp_path / f"{kind}_{len(v)}_{seed}.arpa")
    if kind.startswith("token"):
        LO.write_synthetic_arpa(path, v, order=int(kind[-1]), seed=seed + len(v),
                                per_order=2000 if len(v) >= 1000 else 200)
        return (va.NGramLM.from_arpa(path, v), LO.ArpaLM.from_arpa(path, v),
                dict(lm_weight=TOKEN_WEIGHT))
    constrained = kind == "word_constrained"
    WO.write_synthetic_word_arpa(path, letters_of(v), order=3, seed=seed + len(v),
                                 per_order=2000 if len(v) >= 1000 else 200)
    return (va.WordNGramLM.from_arpa(path, v, lexicon_constrained=constrained),
            WO.WordLM(path, v, lexicon_constrained=constrained), dict(lm_weight=WORD_WEIGHT, word_score=WORD_SCORE))


def ragged_logits(B, L, V, seed):
    """(B, L, V) logits with seeded lengths that include 0, 1 and L, and NaN in every padding row."""
    rs = np.random.RandomState(seed)
    lg = (rs.standard_normal((B, L, V)) * 2.5).astype(np.float32)
    lens = [0, 1, L] + [int(x) for x in rs.randint(2, L, size=B - 3)]
    for b, n in enumerate(lens):
        lg[b, n:] = np.nan
    return torch.from_numpy(lg).cuda(), lens


@pytest.mark.gpu
@pytest.mark.parametrize("V", [40, 1000])
@pytest.mark.parametrize("kind", KINDS)
def test_ragged_equals_each_utterance_alone(va, tmp_path, kind, V):
    v = vocab(V)
    lm, _, kw = make_lm(va, kind, v, tmp_path)
    L = 48 if V == 40 else 96
    lg, lens = ragged_logits(6, L, V, seed=V + len(kind))
    for W in (1, 10, 32):
        got = va.ctc_beam_search(lg, beam_width=W, lm_scorer=lm, lengths=lens, **kw)
        assert len(got) == len(lens)
        for b, n in enumerate(lens):
            alone = va.ctc_beam_search(lg[b:b + 1, :n], beam_width=W, lm_scorer=lm, **kw)[0]
            assert beams_of([got[b]]) == beams_of([alone]), (kind, V, W, b, n)
        assert any(len(d.tokens) > 0 for u in got for d in u)
        # full lengths: exactly the unragged call (on logits without NaN)
        full = lg[[2, 2]]
        assert beams_of(va.ctc_beam_search(full, beam_width=W, lm_scorer=lm, lengths=[L, L], **kw)) == \
            beams_of(va.ctc_beam_search(full, beam_width=W, lm_scorer=lm, **kw))
    # the empty utterance: the single empty beam (under a word LM it carries lm_weight * lm((<s>), </s>))
    assert [d.tokens for d in got[0]] == [[]]
    if kind.startswith("word"):
        assert got[0][0].score == pytest.approx(WORD_WEIGHT * float(lm.log_prob([[]], ["</s>"])[0]), abs=1e-6)
    else:
        assert got[0][0].score == 0.0
    dec = va.CTCDecoder(v)
    assert dec.decode_beam_search(lg, beam_width=10, lm_scorer=lm, lengths=lens, **kw) == \
        [dec.decode_beam_search(lg[b:b + 1, :n], beam_width=10, lm_scorer=lm, **kw)[0] for b, n in enumerate(lens)]
    if lm is not None:
        lm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_ragged_matches_oracle(va, tmp_path, kind):
    v = vocab(40)
    lm, ref, kw = make_lm(va, kind, v, tmp_path, seed=3)
    lg, lens = ragged_logits(5, 30, 40, seed=11)
    got = va.ctc_beam_search(lg, beam_width=10, lm_scorer=lm, lengths=lens, **kw)
    for b, n in enumerate(lens):
        if n == 0:
            continue
        x = lg[b:b + 1, :n].cpu().numpy()
        if kind == "none":
            want = O.ctc_beam_search(x, 10)[0]
        elif kind.startswith("token"):
            want = LO.ctc_beam_search(x, 10, lm_scorer=ref, lm_weight=TOKEN_WEIGHT)[0]
        else:
            want = WO.ctc_beam_search(x, 10, 0, ref, WORD_WEIGHT, WORD_SCORE)[0]
        assert [d.tokens for d in got[b]] == [t for t, _ in want], (kind, b)
        assert np.allclose([d.score for d in got[b]], [s for _, s in want], rtol=0, atol=2e-4), (kind, b)
    if lm is not None:
        lm.close()


SAMPLE_LENS = [16000, 4800, 240000, 96000, 23457, 201 + 160, 240000]   # every pooling branch, odd counts


def make_model(va, mode):
    torch.manual_seed(FU.WEIGHT_SEED)
    m = va.VELOCITYASR(va.VelocityASRConfig(scan_mode=mode))
    m.load_state_dict(FU.amplify_state_dict(m.state_dict()))
    return m.cuda().eval()


def padded_pcm():
    S = max(SAMPLE_LENS)
    g = torch.Generator().manual_seed(5)
    pcm = torch.randn(len(SAMPLE_LENS), S, generator=g) * 0.3             # the padding is noise, not zeros
    for b, n in enumerate(SAMPLE_LENS):
        pcm[b, :n] = FU.synth_audio(1, n, seed=60 + b)[0]
    return pcm


def composed(va, m, pcm, W, lm, kw):
    """The n-best of each utterance alone, through the separate public steps."""
    out = []
    for b, n in enumerate(SAMPLE_LENS):
        logits = m(va.compute_mel_spectrogram(pcm[b, :n].cuda()).unsqueeze(0))
        out.append(va.ctc_beam_search(logits, beam_width=W, lm_scorer=lm, **kw)[0])
    return beams_of(out)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_transcribe_beam_equals_composed(va, tmp_path, mode):
    m = make_model(va, mode)
    v = vocab(m.config.vocab_size)
    pcm = padded_pcm()
    host = pcm.pin_memory()
    for kind in ("none", "token3", "word"):
        lm, _, kw = make_lm(va, kind, v, tmp_path, seed=7)
        want = composed(va, m, pcm, 8, lm, kw)
        assert any(len(t) > 0 for u in want for t, _ in u)
        assert beams_of(m.transcribe_beam(pcm.cuda(), lengths=SAMPLE_LENS, beam_width=8, lm_scorer=lm, **kw)) == want
        assert beams_of(m.transcribe_beam(host, lengths=torch.tensor(SAMPLE_LENS), beam_width=8, lm_scorer=lm,
                                          **kw)) == want
        full = [2, 6]                                                        # utterances that fill all S samples
        for x in (pcm[full].cuda(), host[full]):
            assert beams_of(m.transcribe_beam(x, beam_width=8, lm_scorer=lm, **kw)) == [want[b] for b in full]
        if lm is not None:
            lm.close()
    one = m.transcribe_beam(pcm[0, :SAMPLE_LENS[0]].cuda(), beam_width=3)             # (S,) input
    assert len(one) == 1 and all(d.text == "" for d in one[0])


@pytest.mark.gpu
def test_transcribe_beam_quantized_model(va):
    m = make_model(va, "sequential")
    va.prepare_model_for_qat(m)
    va.calibrate_model(m, [va.compute_mel_spectrogram(FU.synth_audio(2, 16000).cuda())])
    pcm = padded_pcm()
    want = composed(va, m, pcm, 6, None, {})
    assert beams_of(m.transcribe_beam(pcm.cuda(), lengths=SAMPLE_LENS, beam_width=6)) == want
    assert beams_of(m.transcribe_beam(pcm.pin_memory(), lengths=SAMPLE_LENS, beam_width=6)) == want


@pytest.mark.gpu
def test_transcribe_beam_errors(va, tmp_path):
    m = make_model(va, "sequential")
    V = m.config.vocab_size
    v = vocab(V)
    pcm = FU.synth_audio(2, 8000).cuda()
    logits = m(va.compute_mel_spectrogram(pcm))

    def same_error(**kw):
        """transcribe_beam raises what ctc_beam_search raises for the same search arguments."""
        with pytest.raises(Exception) as want:
            va.ctc_beam_search(logits, **kw)
        with pytest.raises(want.type):
            m.transcribe_beam(pcm, **kw)
        with pytest.raises(want.type):
            m.transcribe_beam(pcm.cpu().pin_memory(), **kw)
        return want.type

    p = str(tmp_path / "small.arpa")
    LO.write_synthetic_arpa(p, vocab(40), order=2, seed=1)
    small = va.NGramLM.from_arpa(p, vocab(40))
    assert same_error(lm_scorer=small, lm_weight=1.0) is ValueError                   # another vocabulary size
    p = str(tmp_path / "blank1.arpa")
    LO.write_synthetic_arpa(p, v, order=2, seed=1, blank_token=1)
    blank1 = va.NGramLM.from_arpa(p, v, blank_token=1)
    assert same_error(lm_scorer=blank1, lm_weight=1.0) is ValueError                  # another blank
    p = str(tmp_path / "tok.arpa")
    LO.write_synthetic_arpa(p, v, order=2, seed=1)
    tok = va.NGramLM.from_arpa(p, v)
    assert same_error(lm_scorer=tok, lm_weight=1.0, word_score=1.0) is ValueError
    assert same_error(beam_width=0) is ValueError
    assert same_error(beam_width=33) is ValueError
    for x in (pcm, pcm.cpu().pin_memory()):                                           # checked before any buffer
        with pytest.raises(ValueError, match="beam_width"):
            m.transcribe_beam(x, beam_width=-1)
    assert same_error(lm_scorer=lambda prefix, t: 0.0, lm_weight=1.0) is NotImplementedError
    with pytest.raises(RuntimeError):
        m.transcribe_beam(pcm, lengths=[8000])                                         # wrong count
    with pytest.raises(RuntimeError):
        m.transcribe_beam(pcm, lengths=[8000, 200])                                    # too short for the mel
    if torch.cuda.device_count() > 1:
        other = va.NGramLM.from_arpa(p, v, device=torch.device("cuda", 1))
        assert same_error(lm_scorer=other, lm_weight=1.0) is ValueError
        other.close()
    for lm in (small, blank1, tok):
        lm.close()
