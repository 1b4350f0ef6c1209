"""CTC decoding: ctc_greedy_decode / CTCDecoder / create_default_vocabulary of
velocity_asr/decode.py, with the argmax and the blank/repeat collapse done on the GPU."""
import ctypes
import math
from dataclasses import dataclass
from typing import Any, List, Optional, Tuple

import torch

from . import _native
from .lm import NGramLM, WordNGramLM

BLANK_TOKEN = 0  # decode.py:14


def ctc_greedy_decode(logits: torch.Tensor, blank_token: int = BLANK_TOKEN,
                      collapse_repeated: bool = True) -> List[List[int]]:
    """logits (B, L, V) -> token-id lists.  Same rule as decode.py:46-69: argmax (ties -> lowest index),
    drop blanks, collapse repeats, a blank resets the repeat state.  Runs in the CUDA kernels whatever the
    device of `logits` (CPU logits are copied to the current CUDA device first; no CUDA device -> RuntimeError)."""
    if logits.dim() != 3:
        raise RuntimeError(f"expected (batch, seq_len, vocab) logits, got {tuple(logits.shape)}")
    if logits.device.type != "cuda":       # host logits: staged to the current CUDA device (no CPU decoder exists)
        logits = logits.to(_native.default_cuda_device())
    B, L, V = logits.shape
    if B == 0:
        return []
    if L == 0:
        return [[] for _ in range(B)]
    lg = logits.to(torch.float32).contiguous()
    tokens = torch.empty(B, L, dtype=torch.int32, device=lg.device)
    lens = torch.empty(B, dtype=torch.int32, device=lg.device)
    lib = _native.lib()
    with torch.cuda.device(lg.device):
        _native.check(lib.vasr_ctc_greedy(_native.ptr(lg), B, L, V, int(blank_token), int(bool(collapse_repeated)),
                                          _native.ptr(tokens), _native.ptr(lens),
                                          ctypes.c_void_p(torch.cuda.current_stream(lg.device).cuda_stream)))
    tokens, lens = tokens.cpu(), lens.cpu()
    return [tokens[b, : int(lens[b])].tolist() for b in range(B)]


def ctc_greedy_decode_with_timestamps(logits: torch.Tensor, blank_token: int = BLANK_TOKEN
                                      ) -> List[Tuple[List[int], List[Tuple[int, int]]]]:
    """decode.py:74-125: per utterance (tokens, [(start_frame, end_frame), ...]); a token's range is the run
    of equal non-blank argmax frames it was collapsed from (end exclusive).  Frame -> seconds is
    frame * 2 * 160 / 16000 (scripts/transcribe.py:42-45)."""
    if logits.dim() != 3:
        raise RuntimeError(f"expected (batch, seq_len, vocab) logits, got {tuple(logits.shape)}")
    if logits.device.type != "cuda":       # host logits: staged to the current CUDA device (no CPU decoder exists)
        logits = logits.to(_native.default_cuda_device())
    B, L, V = logits.shape
    if B == 0:
        return []
    if L == 0:
        return [([], []) for _ in range(B)]
    lg = logits.to(torch.float32).contiguous()
    buf = torch.empty(3, B, L, dtype=torch.int32, device=lg.device)
    lens = torch.empty(B, dtype=torch.int32, device=lg.device)
    lib = _native.lib()
    with torch.cuda.device(lg.device):
        _native.check(lib.vasr_ctc_greedy_timestamps(
            _native.ptr(lg), B, L, V, int(blank_token), _native.ptr(buf[0]), _native.ptr(buf[1]), _native.ptr(buf[2]),
            _native.ptr(lens), ctypes.c_void_p(torch.cuda.current_stream(lg.device).cuda_stream)))
    buf, lens = buf.cpu().numpy(), lens.cpu().tolist()
    return [(buf[0, b, :n].tolist(), list(zip(buf[1, b, :n].tolist(), buf[2, b, :n].tolist())))
            for b, n in enumerate(lens)]


@dataclass
class GreedyResult:
    """One utterance's greedy path with scores (include/vasr.h, vasr_ctc_greedy_confidence, states the rule).
    tokens: the greedy transcript.  timestamps: per token its [start, end) frame range (the run of equal non-blank
    argmax frames it was collapsed from).  token_log_probs: per token the sum of its frames' log-softmax values at the
    argmax (fp64).  log_prob: that sum over every frame of the utterance, blank frames included: the log-prob of the
    greedy path (fp64)."""

    tokens: List[int]
    timestamps: List[Tuple[int, int]]
    token_log_probs: List[float]
    log_prob: float


def _greedy_results(buf, tlp, lens, lp) -> List[GreedyResult]:
    """(3, B, L) tokens / starts / ends, (B, L) token log-probs, (B,) lens and (B,) log-probs -> GreedyResult list."""
    buf, tlp, lens, lp = buf.cpu().numpy(), tlp.cpu().numpy(), lens.cpu().tolist(), lp.cpu().tolist()
    return [GreedyResult(tokens=buf[0, b, :n].tolist(), timestamps=list(zip(buf[1, b, :n].tolist(), buf[2, b, :n].tolist())),
                         token_log_probs=tlp[b, :n].tolist(), log_prob=lp[b]) for b, n in enumerate(lens)]


def ctc_greedy_decode_with_confidence(logits: torch.Tensor, lengths=None, blank_token: int = BLANK_TOKEN
                                      ) -> List[GreedyResult]:
    """ctc_greedy_decode_with_timestamps plus scores: per utterance a GreedyResult with the same tokens and
    timestamps, each token's log-prob (the sum over its frames of log_softmax(logits)[argmax], the fp32 table of the
    beam search, added in fp64) and the greedy path's log-prob.  `lengths` (B frame counts in [0, L]): utterance b is
    decoded over its first lengths[b] frames only, bit for bit as if alone.  Host logits are staged to the current
    CUDA device.  A bad length raises RuntimeError, a blank outside the vocabulary ValueError, before device work."""
    if logits.dim() != 3:
        raise RuntimeError(f"expected (batch, seq_len, vocab) logits, got {tuple(logits.shape)}")
    B, L, V = logits.shape
    rows = None
    if lengths is not None:
        from .model import _lengths_tensor
        rows = _lengths_tensor(lengths, B)
        if B and (int(rows.min()) < 0 or int(rows.max()) > L):
            raise RuntimeError(f"every length must be in [0, {L}], got {rows.tolist()}")
    if not 0 <= int(blank_token) < V:
        raise ValueError(f"blank token {blank_token} is outside the vocabulary of {V}")
    if logits.device.type != "cuda":       # host logits: staged to the current CUDA device (no CPU decoder exists)
        logits = logits.to(_native.default_cuda_device())
    if B == 0:
        return []
    lg = logits.to(torch.float32).contiguous()
    buf = torch.empty(3, B, max(L, 1), dtype=torch.int32, device=lg.device)
    tlp = torch.empty(B, max(L, 1), dtype=torch.float64, device=lg.device)
    lens = torch.empty(B, dtype=torch.int32, device=lg.device)
    lp = torch.empty(B, dtype=torch.float64, device=lg.device)
    with torch.cuda.device(lg.device):
        _native.check(_native.lib().vasr_ctc_greedy_confidence(
            _native.ptr(lg), _native.ptr(rows), B, L, V, int(blank_token), _native.ptr(buf[0]), _native.ptr(buf[1]),
            _native.ptr(buf[2]), _native.ptr(tlp), _native.ptr(lens), _native.ptr(lp),
            ctypes.c_void_p(torch.cuda.current_stream(lg.device).cuda_stream)))
    return _greedy_results(buf, tlp, lens, lp)


def frames_to_seconds(frame_idx: int, hop_length: int = 160, sample_rate: int = 16000) -> float:
    """Token index -> seconds (scripts/transcribe.py:42-45): one token spans two mel frames (stride-2 conv)."""
    return (frame_idx * 2 * hop_length) / sample_rate


def words_with_timestamps(tokens: List[int], timestamps: List[Tuple[int, int]], vocabulary: List[str],
                          token_log_probs: Optional[List[float]] = None) -> List[dict]:
    """Word assembly of scripts/transcribe.py:80-126 on one utterance's output of
    ctc_greedy_decode_with_timestamps: characters accumulate into a word until a space / subword marker; a
    word starts at its first character's start frame and ends at the END frame of the separator that closed
    it (the last word: at the end frame of the last token).  Returns [{"word", "start", "end"}] in seconds.
    With token_log_probs (a GreedyResult's), each word also gets "confidence" = exp(sum of its characters' token
    log-probs / sum of their frame counts): the geometric mean of its characters' frame probabilities, separators
    excluded."""
    words, chars, start = [], [], None
    lp_sum, n_frames = 0.0, 0

    def close(end_frame):
        text = "".join(chars).replace("▁", "")
        if text:
            w = {"word": text, "start": frames_to_seconds(start), "end": frames_to_seconds(end_frame)}
            if token_log_probs is not None:
                w["confidence"] = math.exp(lp_sum / n_frames)
            words.append(w)

    for i, (tok, (f0, f1)) in enumerate(zip(tokens, timestamps)):
        ch = vocabulary[tok] if 0 <= tok < len(vocabulary) else "<unk>"
        if ch in (" ", "▁"):
            if chars:
                close(f1)
                chars, start = [], None
                lp_sum, n_frames = 0.0, 0
        else:
            if start is None:
                start = f0
            chars.append(ch)
            if token_log_probs is not None:
                lp_sum += token_log_probs[i]
                n_frames += f1 - f0
    if chars and timestamps:
        close(timestamps[-1][1])
    return words


@dataclass
class DecodingResult:
    """decode.py:17-24."""

    text: str
    tokens: List[int]
    score: float
    timestamps: Optional[List[Tuple[int, int]]] = None


def _search_lm(lm_scorer: Optional[Any], lm_weight: float, word_score: float):
    """The LM rules shared by ctc_beam_search and VELOCITYASR.transcribe_beam: the LM to search with, or None when
    the search runs LM-free (off means off).  A Python `lm_scorer` callback with lm_weight > 0 cannot run inside the
    device loop and is refused rather than silently ignored."""
    word_lm = isinstance(lm_scorer, WordNGramLM)
    if word_lm:
        if not (math.isfinite(lm_weight) and lm_weight >= 0):
            raise ValueError(f"lm_weight must be finite and >= 0 with a WordNGramLM, got {lm_weight}")
        if not math.isfinite(word_score):
            raise ValueError(f"word_score must be finite, got {word_score}")
        use_lm = lm_weight != 0 or word_score != 0 or lm_scorer.lexicon_constrained
    else:
        if word_score != 0:
            raise ValueError("word_score needs a WordNGramLM as lm_scorer")
        use_lm = isinstance(lm_scorer, NGramLM) and lm_weight > 0
    if lm_scorer is not None and lm_weight > 0 and not use_lm:
        raise NotImplementedError("velocity_asr (B200 build): ctc_beam_search runs on the device and takes no "
                                  "Python lm_scorer (use velocity_asr.NGramLM)")
    return lm_scorer if use_lm else None


def _check_lm_fits(lm, V: int, blank_token: int) -> None:
    lm._live()
    if V != lm.vocab_size:
        raise ValueError(f"the LM is built for a vocabulary of {lm.vocab_size} tokens, the logits have {V}")
    if int(blank_token) != lm.blank_token:
        raise ValueError(f"the LM is built with blank token {lm.blank_token}, the search uses {blank_token}")


def _beam_results(tokens: torch.Tensor, lens: torch.Tensor, scores: torch.Tensor) -> List[List[DecodingResult]]:
    """(B, W, L) tokens, (B, W) lens (-1: no such beam), (B, W) fp64 scores -> per utterance its beams, best first."""
    tokens, lens, scores = tokens.cpu().numpy(), lens.cpu().tolist(), scores.cpu().tolist()
    return [[DecodingResult(text="", tokens=tokens[b, r, :n].tolist(), score=scores[b][r])
             for r, n in enumerate(lens[b]) if n >= 0] for b in range(len(lens))]


def ctc_beam_search(logits: torch.Tensor, beam_width: int = 10, blank_token: int = BLANK_TOKEN,
                    lm_weight: float = 0.0, lm_scorer: Optional[Any] = None,
                    word_score: float = 0.0, lengths=None) -> List[List[DecodingResult]]:
    """decode.py:128-217 on the GPU: per utterance the `beam_width` best prefixes, best first, with the
    reference's rule (log_softmax; blank / repeated token keep the prefix, any other token extends it; equal
    prefixes keep the better score; fp64 score sums; ties in insertion order).

    Shallow fusion: with an NGramLM as `lm_scorer` and lm_weight > 0, an offer that extends a prefix by `tok`
    scores (score + log_prob[tok]) + lm_weight * lm(prefix, tok); blank and repeat offers are unchanged and the
    returned scores are the fused ones.  The LM must be built for this vocabulary size and blank token and live on
    the logits' device (host logits are staged to it).  A Python `lm_scorer` callback cannot run inside the device
    loop and is refused rather than silently ignored.

    With a WordNGramLM, words are spelled in the vocabulary and closed by its delimiter: closing a non-empty word
    adds lm_weight * lm(history, word) + word_score, and the end of the utterance closes the last word and adds
    lm_weight * lm(history, </s>) (include/vasr.h states the rule).  lm_weight must be finite and >= 0 and
    word_score finite.  A lexicon-free word LM with lm_weight == 0 and word_score == 0 takes the plain search; in
    lexicon-constrained mode beams that cannot end on a lexicon word are dropped, so fewer may come back.

    `lengths` (B frame counts, each in [0, L]; a list, tuple or tensor): a ragged batch, such as the logits of
    forward(mel, lengths=...).  Utterance b is searched over its first lengths[b] frames only and gets bit for bit
    what ctc_beam_search(logits[b:b+1, :lengths[b]]) gives; the padding rows are never read.  A wrong count or a
    length outside [0, L] raises RuntimeError before any device work."""
    lm = _search_lm(lm_scorer, lm_weight, word_score)
    if logits.dim() != 3:
        raise RuntimeError(f"expected (batch, seq_len, vocab) logits, got {tuple(logits.shape)}")
    B, L, V = logits.shape
    rows = None
    if lengths is not None:
        from .model import _lengths_tensor
        rows = _lengths_tensor(lengths, B)
        if B and (int(rows.min()) < 0 or int(rows.max()) > L):
            raise RuntimeError(f"every length must be in [0, {L}], got {rows.tolist()}")
    if lm is not None:
        _check_lm_fits(lm, V, blank_token)
        if logits.device.type != "cuda":   # host logits: staged to the LM's device
            logits = logits.to(lm.device)
        elif logits.device != lm.device:
            raise ValueError(f"the LM is on {lm.device}, the logits on {logits.device}")
    elif logits.device.type != "cuda":     # host logits: staged to the current CUDA device (no CPU decoder exists)
        logits = logits.to(_native.default_cuda_device())
    W = int(beam_width)
    if B == 0:
        return []
    lg = logits.to(torch.float32).contiguous()
    tokens = torch.empty(B, W, max(L, 1), dtype=torch.int32, device=lg.device)
    lens = torch.empty(B, W, dtype=torch.int32, device=lg.device)
    scores = torch.empty(B, W, dtype=torch.float64, device=lg.device)
    with torch.cuda.device(lg.device):
        _native.check(_native.lib().vasr_ctc_beam_search_ragged(
            _native.ptr(lg), _native.ptr(rows), B, L, V, W, int(blank_token), lm._handle if lm is not None else None,
            float(lm_weight), float(word_score), _native.ptr(tokens), _native.ptr(lens), _native.ptr(scores),
            ctypes.c_void_p(torch.cuda.current_stream(lg.device).cuda_stream)))
    return _beam_results(tokens, lens, scores)


@dataclass
class AlignmentResult:
    """One utterance's CTC forced alignment (include/vasr.h, vasr_ctc_align, states the rule).
    tokens: the target.  timestamps: per token its [start, end) frame range on the best path, or None when the
    target cannot fit.  frame_labels (frames,) int32 / frame_log_probs (frames,) float32 host tensors over the
    utterance's own frames: the label of the state the best path occupies at each frame (blank included) and the
    log-prob there; -1 / 0 everywhere when there is no path.  score: the best path's log-prob, fp64 (-inf: no path)."""

    tokens: List[int]
    timestamps: Optional[List[Tuple[int, int]]]
    frame_labels: torch.Tensor
    frame_log_probs: torch.Tensor
    score: float


def _align_targets(targets, B: int, V: int, blank_token: int):
    """Token-id lists -> (host int32 (B, max(U_max, 1)) targets, host int32 (B,) lengths, U_max).  Raises before any
    device work: RuntimeError for a count that is not B, ValueError for a blank outside the vocabulary or an id
    outside it or equal to the blank."""
    import numpy as np
    if len(targets) != B:
        raise RuntimeError(f"expected {B} targets, got {len(targets)}")
    if not 0 <= int(blank_token) < V:
        raise ValueError(f"blank token {blank_token} is outside the vocabulary of {V}")
    rows = [np.asarray(t, dtype=np.int64).reshape(-1) for t in targets]
    U_max = max((r.size for r in rows), default=0)
    tgt = np.zeros((B, max(U_max, 1)), np.int32)
    for b, r in enumerate(rows):
        if r.size and (r.min() < 0 or r.max() >= V or (r == blank_token).any()):
            raise ValueError(f"target {b} has an id outside [0, {V}) or equal to the blank {blank_token}")
        tgt[b, :r.size] = r
    return torch.from_numpy(tgt), torch.tensor([r.size for r in rows], dtype=torch.int32), U_max


def _alignment_results(tgt: torch.Tensor, tlens: torch.Tensor, labels: torch.Tensor, lps: torch.Tensor,
                       scores: torch.Tensor, frames: List[int], blank_token: int) -> List[AlignmentResult]:
    """The targets and lengths of _align_targets, (B, L) labels / log-probs and (B,) scores of vasr_ctc_align -> one
    AlignmentResult per utterance."""
    labels, lps, scores = labels.cpu(), lps.cpu(), scores.cpu().tolist()
    tgt, tlens = tgt.numpy(), tlens.tolist()
    # equal neighbouring targets are separated by a blank on every path, so a run of one label is one token; frames
    # without a path or past an utterance's end are -1.  Runs are found for the whole batch at once.
    x = labels.numpy()[:, :max(frames, default=0)]
    tok = (x != blank_token) & (x >= 0)
    start = tok.copy()
    start[:, 1:] &= x[:, 1:] != x[:, :-1]
    end = tok.copy()
    end[:, :-1] &= x[:, :-1] != x[:, 1:]
    starts = start.nonzero()[1].tolist()
    ends = (end.nonzero()[1] + 1).tolist()
    out, k = [], 0
    for b, n in enumerate(frames):                       # a path has one run per token; no path has none
        m = tlens[b] if scores[b] != -math.inf else 0
        spans = list(zip(starts[k:k + m], ends[k:k + m])) if scores[b] != -math.inf else None
        k += m
        out.append(AlignmentResult(tokens=tgt[b, :tlens[b]].tolist(), timestamps=spans, frame_labels=labels[b, :n],
                                   frame_log_probs=lps[b, :n], score=scores[b]))
    return out


def _align_inputs(logits: torch.Tensor, targets, lengths, blank_token: int):
    """Checks and staging shared by ctc_forced_align and ctc_log_likelihood (all checks before device work)."""
    if logits.dim() != 3:
        raise RuntimeError(f"expected (batch, seq_len, vocab) logits, got {tuple(logits.shape)}")
    B, L, V = logits.shape
    tgt, tlens, U_max = _align_targets(targets, B, V, blank_token)
    rows = None
    if lengths is not None:
        from .model import _lengths_tensor
        rows = _lengths_tensor(lengths, B)
        if B and (int(rows.min()) < 0 or int(rows.max()) > L):
            raise RuntimeError(f"every length must be in [0, {L}], got {rows.tolist()}")
    if logits.device.type != "cuda":       # host logits: staged to the current CUDA device (no CPU path exists)
        logits = logits.to(_native.default_cuda_device())
    frames = [L] * B if rows is None else rows.tolist()
    return logits.to(torch.float32).contiguous(), rows, tgt, tlens, U_max, frames


def ctc_forced_align(logits: torch.Tensor, targets: List[List[int]], lengths=None, blank_token: int = BLANK_TOKEN,
                     log_probs: bool = False) -> List[AlignmentResult]:
    """CTC forced alignment on the GPU: per utterance the best path of its target (a list of token ids) through its
    logits (B, L, V), with each token's [start, end) frame range (the units of ctc_greedy_decode_with_timestamps).
    Per-frame log-probs are log_softmax(logits) in fp32, as the beam search computes them, or the input itself with
    log_probs=True; path scores are fp64.  Ties go to the earlier of stay / advance / skip and, at the end, to the
    last-token state (include/vasr.h states the rule).  `lengths` (B frame counts in [0, L]): utterance b is aligned
    over its first lengths[b] frames only, bit for bit as if alone.  Host logits are staged to the current CUDA
    device.  A bad id raises ValueError, a bad length RuntimeError, both before any device work."""
    lg, rows, tgt, tlens, U_max, frames = _align_inputs(logits, targets, lengths, blank_token)
    B, L, V = lg.shape
    if B == 0:
        return []
    labels = torch.empty(B, max(L, 1), dtype=torch.int32, device=lg.device)
    lps = torch.empty(B, max(L, 1), dtype=torch.float32, device=lg.device)
    scores = torch.empty(B, dtype=torch.float64, device=lg.device)
    with torch.cuda.device(lg.device):
        _native.check(_native.lib().vasr_ctc_align(
            _native.ptr(lg), _native.ptr(rows), B, L, V, int(blank_token), int(bool(log_probs)), _native.ptr(tgt),
            _native.ptr(tlens), U_max, _native.ptr(labels), _native.ptr(lps), _native.ptr(scores),
            ctypes.c_void_p(torch.cuda.current_stream(lg.device).cuda_stream)))
    return _alignment_results(tgt, tlens, labels, lps, scores, frames, int(blank_token))


def ctc_log_likelihood(logits: torch.Tensor, targets: List[List[int]], lengths=None, blank_token: int = BLANK_TOKEN,
                       log_probs: bool = False) -> torch.Tensor:
    """log P(target | logits) under CTC, summed over every alignment, per utterance: (B,) float64, equal to
    -torch.nn.functional.ctc_loss(..., reduction="none") (-inf when the target cannot fit).  Arguments, checks and
    staging as ctc_forced_align; the result is on the logits' device."""
    home = logits.device
    lg, rows, tgt, tlens, U_max, _ = _align_inputs(logits, targets, lengths, blank_token)
    B, L, V = lg.shape
    ll = torch.empty(B, dtype=torch.float64, device=lg.device)
    if B > 0:
        with torch.cuda.device(lg.device):
            _native.check(_native.lib().vasr_ctc_log_likelihood(
                _native.ptr(lg), _native.ptr(rows), B, L, V, int(blank_token), int(bool(log_probs)),
                _native.ptr(tgt), _native.ptr(tlens), U_max, _native.ptr(ll),
                ctypes.c_void_p(torch.cuda.current_stream(lg.device).cuda_stream)))
    return ll if home.type == "cuda" else ll.to(home)


class CTCDecoder:
    """decode.py:220-328: vocabulary lookup around the greedy and beam-search decoders."""

    def __init__(self, vocabulary: List[str], blank_token: int = BLANK_TOKEN):
        self.vocabulary = vocabulary
        self.blank_token = blank_token
        self.vocab_size = len(vocabulary)
        self.token_to_idx = {tok: i for i, tok in enumerate(vocabulary)}

    def decode_greedy(self, logits: torch.Tensor, collapse_repeated: bool = True) -> List[str]:
        seqs = ctc_greedy_decode(logits, blank_token=self.blank_token, collapse_repeated=collapse_repeated)
        return [self._tokens_to_text(s) for s in seqs]

    def decode_beam_search(self, logits: torch.Tensor, beam_width: int = 10, return_all_beams: bool = False,
                           lm_scorer: Optional[Any] = None, lm_weight: float = 0.0, word_score: float = 0.0,
                           lengths=None):
        """decode.py:265-300: best-beam texts, or every beam with its text filled in.  `lm_scorer` / `lm_weight` /
        `word_score` / `lengths` go to ctc_beam_search (shallow fusion with an NGramLM or a WordNGramLM; a ragged
        batch)."""
        beams = ctc_beam_search(logits, beam_width=beam_width, blank_token=self.blank_token, lm_weight=lm_weight,
                                lm_scorer=lm_scorer, word_score=word_score, lengths=lengths)
        if return_all_beams:
            for utt in beams:
                for r in utt:
                    r.text = self._tokens_to_text(r.tokens)
            return beams
        return [self._tokens_to_text(utt[0].tokens) if utt else "" for utt in beams]

    def align(self, logits: torch.Tensor, texts: List[str], lengths=None) -> List[List[dict]]:
        """Word timings of known transcripts: each text goes through text_to_tokens, is force-aligned to its logits
        (ctc_forced_align) and assembled into words by words_with_timestamps ([{"word", "start", "end"}] in
        seconds).  A transcript that cannot fit its frames gives []."""
        res = ctc_forced_align(logits, [self.text_to_tokens(t) for t in texts], lengths=lengths,
                               blank_token=self.blank_token)
        return [words_with_timestamps(r.tokens, r.timestamps, self.vocabulary) if r.timestamps is not None else []
                for r in res]

    def _tokens_to_text(self, tokens: List[int]) -> str:
        """decode.py:302-317: join, then turn the subword marker into spaces."""
        pieces = [self.vocabulary[t] if 0 <= t < self.vocab_size else "<unk>" for t in tokens]
        return "".join(pieces).replace("▁", " ").strip()

    def text_to_tokens(self, text: str) -> List[int]:
        unk = self.token_to_idx.get("<unk>")
        out = []
        for ch in text:
            if ch in self.token_to_idx:
                out.append(self.token_to_idx[ch])
            elif unk is not None:
                out.append(unk)
        return out


def create_default_vocabulary(vocab_size: int = 50000) -> List[str]:
    """decode.py:330-362: specials, space, a-z, A-Z, 0-9, punctuation, then <token_i> fillers."""
    import string
    vocab = ["<blank>", "<unk>", "<pad>", " "]
    vocab += list(string.ascii_lowercase) + list(string.ascii_uppercase) + list(string.digits)
    vocab += list(".,!?;:'\"()-")
    vocab += [f"<token_{i}>" for i in range(len(vocab), vocab_size)]
    return vocab
