"""N-gram language models for shallow fusion in the device prefix beam search (ctc_beam_search(lm_scorer=...)).

An ARPA file is read by libvasr's C++ parser and kept as device tables; nothing here loops over the file.
NGramLM scores token ids; WordNGramLM scores words spelled in a character vocabulary and closed by a delimiter.
Both use standard ARPA back-off in natural log (include/vasr.h states the exact rules)."""
import ctypes
import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native


def _device_index(device, what):
    if device is None:
        return -1
    device = torch.device(device)
    if device.type != "cuda":
        raise ValueError(f"{what} lives on a CUDA device, not {device}")
    return device.index if device.index is not None else -1


class _DeviceLM:
    """The native handle and device of an LM; close() (or collection) releases the tables."""

    def __init__(self, handle: ctypes.c_void_p, vocab_size: int, blank_token: int, device: torch.device):
        self._handle = handle
        self.vocab_size = vocab_size
        self.blank_token = blank_token
        self.device = device
        self.order = int(_native.lib().vasr_lm_order(handle))

    def _score(self, prefixes: Sequence[Sequence[int]], symbols: Sequence[int], n_symbols: int) -> torch.Tensor:
        """lm(prefixes[i], symbols[i]) through the scoring kernel; ids in [0, n_symbols)."""
        self._live()
        n = len(symbols)
        if len(prefixes) != n:
            raise ValueError(f"{len(prefixes)} prefixes for {n} tokens")
        H = max(self.order - 1, 1)
        hist = np.zeros((n, H), np.int32)
        lens = np.zeros(n, np.int32)
        for i, pre in enumerate(prefixes):
            pre = list(pre)
            tail = pre[len(pre) - min(len(pre), self.order - 1):] if self.order > 1 else []
            if tail:
                hist[i, H - len(tail):] = tail
            lens[i] = len(pre)
        tok = np.asarray(symbols, np.int64).reshape(n)
        if n and (tok.min() < 0 or tok.max() >= n_symbols or
                  (hist.size and (hist.min() < 0 or hist.max() >= n_symbols))):
            raise ValueError(f"token ids must be in [0, {n_symbols})")
        out = torch.empty(n, dtype=torch.float32, device=self.device)
        if n == 0:
            return out
        d_hist = torch.from_numpy(hist).to(self.device)
        d_lens = torch.from_numpy(lens).to(self.device)
        d_tok = torch.from_numpy(tok.astype(np.int32)).to(self.device)
        with torch.cuda.device(self.device):
            _native.check(_native.lib().vasr_lm_log_prob(
                self._handle, _native.ptr(d_hist), _native.ptr(d_lens), n, _native.ptr(d_tok), _native.ptr(out),
                ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out

    def close(self) -> None:
        if getattr(self, "_handle", None):
            _native.lib().vasr_lm_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _live(self):
        if not self._handle:
            raise RuntimeError(f"{type(self).__name__} is closed")
        return self._handle


class NGramLM(_DeviceLM):
    """A device-resident ARPA n-gram LM over the token ids of `vocabulary`.

    Build it with NGramLM.from_arpa; pass it to ctc_beam_search / CTCDecoder.decode_beam_search as `lm_scorer`
    with lm_weight > 0.  The native tables are released by close() (or when the object is collected)."""

    @classmethod
    def from_arpa(cls, path, vocabulary: Sequence[str], blank_token: int = 0,
                  device: Optional[torch.device] = None) -> "NGramLM":
        """Parse an ARPA file for `vocabulary` (a word maps to the entry with the same string, <space> to " ") and
        upload it to `device` (default: the current CUDA device).  A malformed file, an order above 8, or a
        non-blank token without a unigram in a file without <unk> raises ValueError naming the line."""
        path = os.fspath(path)
        if not os.path.isfile(path):
            raise FileNotFoundError(path)
        V = len(vocabulary)
        if not 0 <= blank_token < V:
            raise ValueError(f"blank_token {blank_token} is outside the vocabulary of {V} entries")
        index = _device_index(device, "NGramLM")
        words = (ctypes.c_char_p * V)(*[str(w).encode("utf-8") for w in vocabulary])
        handle = ctypes.c_void_p()
        lib = _native.lib()
        _native.check(lib.vasr_lm_create_arpa(path.encode(), words, V, int(blank_token), index,
                                              ctypes.byref(handle)))
        if index < 0:
            index = torch.cuda.current_device()
        return cls(handle, V, int(blank_token), torch.device("cuda", index))

    def log_prob(self, prefixes: Sequence[Sequence[int]], tokens: Sequence[int]) -> torch.Tensor:
        """lm(prefixes[i], tokens[i]) for every i, fp32 on the LM's device: the log-probability the beam search adds
        (times lm_weight) when it extends prefixes[i] by tokens[i]; summed over a sequence, it rescores n-best lists."""
        return self._score(prefixes, tokens, self.vocab_size)


class WordNGramLM(_DeviceLM):
    """A device-resident word-level ARPA n-gram LM for a character vocabulary.

    Words are spelled one vocabulary entry per character and closed by `word_delimiter`; the search charges
    lm_weight * lm(history, word) + word_score when a word is closed and lm_weight * lm(history, </s>) at the end of
    the utterance.  With lexicon_constrained=True a hypothesis may only spell words of the lexicon (the LM's
    spellable words).  Build it with WordNGramLM.from_arpa and pass it to ctc_beam_search /
    CTCDecoder.decode_beam_search as `lm_scorer`."""

    def __init__(self, handle, vocab_size, blank_token, device, word_delimiter, lexicon_constrained):
        super().__init__(handle, vocab_size, blank_token, device)
        self.word_delimiter = word_delimiter
        self.lexicon_constrained = lexicon_constrained
        self.lexicon_size = int(_native.lib().vasr_lm_lexicon_size(handle))

    @classmethod
    def from_arpa(cls, path, vocabulary: Sequence[str], blank_token: int = 0, word_delimiter: str = " ",
                  lexicon_constrained: bool = False, device: Optional[torch.device] = None) -> "WordNGramLM":
        """Parse a word-level ARPA file, build its lexicon over `vocabulary` and upload both to `device` (default:
        the current CUDA device).  ValueError, before any device work, for a delimiter missing from the vocabulary
        or equal to the blank, a malformed file (naming the line), lexicon-free mode without <unk>, or constrained
        mode with no spellable word."""
        path = os.fspath(path)
        if not os.path.isfile(path):
            raise FileNotFoundError(path)
        V = len(vocabulary)
        if not 0 <= blank_token < V:
            raise ValueError(f"blank_token {blank_token} is outside the vocabulary of {V} entries")
        index = _device_index(device, "WordNGramLM")
        words = (ctypes.c_char_p * V)(*[str(w).encode("utf-8") for w in vocabulary])
        handle = ctypes.c_void_p()
        lib = _native.lib()
        _native.check(lib.vasr_lm_create_word_arpa(path.encode(), words, V, int(blank_token),
                                                   str(word_delimiter).encode("utf-8"), int(bool(lexicon_constrained)),
                                                   index, ctypes.byref(handle)))
        if index < 0:
            index = torch.cuda.current_device()
        return cls(handle, V, int(blank_token), torch.device("cuda", index), str(word_delimiter),
                   bool(lexicon_constrained))

    def word_ids(self, words: Sequence[str]) -> np.ndarray:
        """The LM's id of each word; a string that is not a word of the LM maps to <unk>."""
        n = len(words)
        ids = np.zeros(n, np.int32)
        if n:
            arr = (ctypes.c_char_p * n)(*[str(w).encode("utf-8") for w in words])
            _native.check(_native.lib().vasr_lm_word_ids(self._live(), arr, n, ids.ctypes.data_as(ctypes.c_void_p)))
        return ids

    def log_prob(self, histories: Sequence[Sequence[str]], words: Sequence[str]) -> torch.Tensor:
        """lm(histories[i], words[i]) for every i, fp32 on the LM's device.  A history is the words after <s>;
        words[i] may be "</s>"; strings the LM does not know score as <unk>.  Summed over a word sequence and its
        closing </s>, it rescores n-best lists with the weights the search uses."""
        self._live()
        if len(histories) != len(words):
            raise ValueError(f"{len(histories)} histories for {len(words)} words")
        flat = self.word_ids([w for h in histories for w in h])
        hist, at = [], 0
        for h in histories:
            hist.append(flat[at:at + len(h)].tolist())
            at += len(h)
        return self._score(hist, self.word_ids(list(words)).tolist(), 2 ** 31 - 1)
