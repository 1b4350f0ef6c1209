"""N-gram language model for shallow fusion in the device prefix beam search (ctc_beam_search(lm_scorer=...)).

An ARPA file is read by libvasr's C++ parser and kept as device tables; nothing here loops over the file.
lm(prefix, tok) is standard ARPA back-off in natural log over token ids (include/vasr.h states the exact rule)."""
import ctypes
import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native


class NGramLM:
    """A device-resident ARPA n-gram LM over the token ids of `vocabulary`.

    Build it with NGramLM.from_arpa; pass it to ctc_beam_search / CTCDecoder.decode_beam_search as `lm_scorer`
    with lm_weight > 0.  The native tables are released by close() (or when the object is collected)."""

    def __init__(self, handle: ctypes.c_void_p, vocab_size: int, blank_token: int, device: torch.device):
        self._handle = handle
        self.vocab_size = vocab_size
        self.blank_token = blank_token
        self.device = device
        self.order = int(_native.lib().vasr_lm_order(handle))

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
        index = -1
        if device is not None:
            device = torch.device(device)
            if device.type != "cuda":
                raise ValueError(f"NGramLM lives on a CUDA device, not {device}")
            index = device.index if device.index is not None else -1
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
        self._live()
        n = len(tokens)
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
        tok = np.asarray(tokens, np.int64).reshape(n)
        if n and (tok.min() < 0 or tok.max() >= self.vocab_size or
                  (hist.size and (hist.min() < 0 or hist.max() >= self.vocab_size))):
            raise ValueError(f"token ids must be in [0, {self.vocab_size})")
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
            raise RuntimeError("NGramLM is closed")
        return self._handle
