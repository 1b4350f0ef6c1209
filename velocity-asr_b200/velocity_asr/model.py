"""VELOCITYASR — the reference's model class (velocity_asr/model.py:242-471) as a thin host
object: parameters live in a torch module tree with the reference's state_dict keys; forward()
runs entirely in libvasr.so (hand-written sm_100a kernels) through the C ABI."""
import ctypes
import os
from typing import Dict, Iterable, Iterator, List, Optional, Tuple, Union

import torch
import torch.nn as nn

from . import _native
from .config import SCAN_MODES, VelocityASRConfig
from .params import build_parameter_tree, reference_init_, time_table


def _stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _token_lists(tokens: torch.Tensor, lens: torch.Tensor) -> List[List[int]]:
    """(B, L) left-packed int32 ids + (B,) counts (host tensors) -> ragged Python lists."""
    # the cost is the creation of the Python ints themselves (~16 k per batch of 64 x 15 s: 0.5 ms); a masked
    # gather + one tolist + slicing was measured slower than per-utterance tolist
    tok = tokens.numpy()
    return [tok[b, :n].tolist() for b, n in enumerate(lens.tolist())]


def _lengths_tensor(lengths, B: int) -> torch.Tensor:
    """Per-utterance lengths (list / tuple / tensor) -> contiguous host int32 tensor of B entries."""
    t = torch.as_tensor(lengths).detach().to("cpu", torch.int32).contiguous().reshape(-1)
    if t.numel() != B:
        raise RuntimeError(f"expected {B} lengths, got {t.numel()}")
    return t


class _Engine:
    """Owns one vasr_handle (one GPU).  Re-uploads weights when the parameters change."""

    @staticmethod
    def config_key(cfg: VelocityASRConfig) -> tuple:
        """The config fields the native handle is created from: a change of any of them (e.g. scan_mode
        edited after the first call) makes VELOCITYASR._engine build a new handle."""
        return (cfg.mel_bins, cfg.d_model, cfg.ssm_layers, cfg.ssm_state_dim, cfg.ssm_expand_ratio,
                cfg.ssm_kernel_size, cfg.global_ssm_layers, cfg.global_ssm_state_dim, cfg.attention_heads,
                cfg.attention_dim, cfg.vocab_size, cfg.scan_mode)

    def __init__(self, cfg: VelocityASRConfig, device: torch.device):
        self.device = device
        self.cfg_key = self.config_key(cfg)
        self.lib = _native.lib()
        c = _native.VasrConfig(
            cfg.mel_bins, cfg.d_model, cfg.ssm_layers, cfg.ssm_state_dim, cfg.ssm_expand_ratio,
            cfg.ssm_kernel_size, cfg.global_ssm_layers, cfg.global_ssm_state_dim, cfg.attention_heads,
            cfg.attention_dim, cfg.vocab_size, _native.SCAN_MODE_ID[cfg.scan_mode])
        self.handle = ctypes.c_void_p()
        _native.check(self.lib.vasr_create(ctypes.byref(c), device.index or 0, ctypes.byref(self.handle)))
        self.fingerprint = None

    def close(self):
        if getattr(self, "handle", None) and self.handle.value:
            self.lib.vasr_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def sync_weights(self, state: Dict[str, torch.Tensor], extra: Dict[str, torch.Tensor], quantized: bool = False,
                     act_qparams: Optional[Dict[str, Tuple[float, float]]] = None):
        # Fingerprint = identity, in-place version counter and shape of every tensor, plus what else shapes
        # the committed weights.  Contract: edits that bypass the version counter (p.data.copy_(), .data.mul_(),
        # EMA updates through .data) are NOT seen — call VELOCITYASR.refresh_weights() after such an edit.
        qp = tuple(sorted((act_qparams or {}).items())) if quantized else ()
        fp = (quantized, qp) + tuple((v.data_ptr(), v._version) for v in state.values())
        fp += tuple((v.data_ptr(), v._version) for v in extra.values())
        if fp == self.fingerprint:
            return
        _native.check(self.lib.vasr_set_quantization(self.handle, int(quantized)))
        for k, v in list(state.items()) + list(extra.items()):
            host = v.detach().to("cpu", torch.float32).contiguous()
            _native.check(self.lib.vasr_set_weight(self.handle, k.encode(), _native.ptr(host), host.numel()))
        _native.check(self.lib.vasr_commit_weights(self.handle))
        for name, (scale, zp) in ((act_qparams or {}) if quantized else {}).items():   # calibration survives a re-commit
            _native.check(self.lib.vasr_set_quant_params(self.handle, name.encode(), scale, zp))
        self.fingerprint = fp


class VELOCITYASR(nn.Module):
    """Drop-in for velocity_asr.VELOCITYASR (model.py:242).  Same constructor, state_dict,
    forward(mel, return_features), get_output_length, from_pretrained / save_pretrained,
    count_parameters; plus transcribe(audio) for the fused PCM -> tokens path.

    Inference only (the reference's callers run it under eval() + no_grad(),
    scripts/transcribe.py:76,225); dropout is the identity.  All arithmetic runs in the CUDA kernels: there is
    no CPU path.  Host tensors are accepted the way the reference's own scripts pass them (test_vel.py:24-37
    never moves model or input off the CPU): they are copied to a CUDA device (the model's, else the current
    one), the kernels run there, and the result is copied back to the input's device.
    """

    def __init__(self, config: Optional[VelocityASRConfig] = None):
        super().__init__()
        if config is None:
            config = VelocityASRConfig()
        if config.scan_mode not in SCAN_MODES:
            raise ValueError(f"Unknown scan_mode: {config.scan_mode}")
        self.config = config
        build_parameter_tree(self, config)
        reference_init_(self)
        self._engines: Dict[int, _Engine] = {}

    # ---- native plumbing ------------------------------------------------------------------
    def _device(self) -> torch.device:
        return self.temporal_binding.conv.weight.device

    def _exec_device(self, like: Optional[torch.Tensor] = None) -> torch.device:
        """Where the kernels run: the input's CUDA device, else the model's, else the current CUDA device."""
        if like is not None and like.device.type == "cuda":
            return like.device
        dev = self._device()
        return dev if dev.type == "cuda" else _native.default_cuda_device()

    def refresh_weights(self) -> None:
        """Forget the device copies of the weights: the next call re-uploads them.  Needed only after edits
        that bypass torch's version counter (p.data.copy_(), .data.mul_(), EMA through .data)."""
        self.__dict__["_state_slots"] = None
        for eng in self._engines.values():
            eng.fingerprint = None

    def _engine(self, device: torch.device) -> _Engine:
        if device.type != "cuda":
            device = self._exec_device()
        if self.config.scan_mode not in SCAN_MODES:
            raise ValueError(f"Unknown scan_mode: {self.config.scan_mode}")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        device = torch.device("cuda", idx)
        eng = self._engines.get(idx)
        if eng is not None and eng.cfg_key != _Engine.config_key(self.config):
            eng.close()                     # the config changed under the handle (e.g. scan_mode): rebuild it
            eng = None
        if eng is None:
            eng = _Engine(self.config, device)
            self._engines[idx] = eng
        from .audio import frontend_tables
        fb, win = frontend_tables(self.config.mel_bins)
        # Same keys and order as state_dict().  The walk over the module tree is cached as (key, owning dict, name)
        # triples (208 tensors: 0.4 ms per call otherwise); the tensors themselves are looked up on every call, so a
        # replaced Parameter object, .to() / .cuda() (new storage) and in-place edits (version counter) are all seen.
        slots = self.__dict__.get("_state_slots")
        if slots is None:
            slots = []
            for prefix, mod in self.named_modules():
                dot = prefix + "." if prefix else ""
                slots += [(dot + n, mod._parameters, n) for n, p in mod._parameters.items() if p is not None]
            for prefix, mod in self.named_modules():
                dot = prefix + "." if prefix else ""
                slots += [(dot + n, mod._buffers, n) for n, b in mod._buffers.items()
                          if b is not None and n not in mod._non_persistent_buffers_set]
            self.__dict__["_state_slots"] = slots
        state = {key: owner[name] for key, owner, name in slots}
        eng.sync_weights(state, {"frontend.mel_filterbank": fb, "frontend.window": win},
                         quantized=getattr(self, "_quantized", False), act_qparams=getattr(self, "_act_qparams", None))
        return eng

    @property
    def _non_persistent(self):
        names = set()
        for m in self.modules():
            names |= set(getattr(m, "_non_persistent_buffers_set", ()))
        return names

    def _check_input(self, x: torch.Tensor, what: str) -> torch.Tensor:
        if not isinstance(x, torch.Tensor):
            raise TypeError(f"{what} must be a torch.Tensor")
        dev = self._device()
        if x.device.type == "cuda" and dev.type == "cuda" and (x.device.index or 0) != (dev.index or 0):
            raise RuntimeError(f"{what} is on {x.device} but the model is on {dev}")
        if x.device.type != "cuda":         # host input: staged to the execution device (see the class docstring)
            x = x.to(self._exec_device())
        return x.to(torch.float32).contiguous()

    # ---- reference API ----------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, mel_spectrogram: torch.Tensor, return_features: bool = False, lengths=None
                ) -> Union[torch.Tensor, Tuple[torch.Tensor, Dict[str, torch.Tensor]]]:
        """(B, T, mel_bins) -> logits (B, (T+1)//2, vocab) [, features].  model.py:333-368.
        `lengths` (B frame counts; not in the reference, whose collator pads and never masks): utterance b
        has lengths[b] valid frames and its logits rows [: get_output_length(lengths[b])] equal those of
        forward(mel[b:b+1, :lengths[b]]); rows past that are padding."""
        home = mel_spectrogram.device if isinstance(mel_spectrogram, torch.Tensor) else None
        mel = self._check_input(mel_spectrogram, "mel_spectrogram")
        back = (lambda t: t) if home is None or home.type == "cuda" else (lambda t: t.to(home))
        if mel.dim() != 3 or mel.size(2) != self.config.mel_bins:
            raise RuntimeError(f"expected (batch, frames, {self.config.mel_bins}) input, got {tuple(mel.shape)}")
        eng = self._engine(mel.device)
        B, T, _ = mel.shape
        L = self.get_output_length(T)
        logits = torch.empty(B, L, self.config.vocab_size, device=mel.device, dtype=torch.float32)
        if lengths is not None:
            if return_features:
                raise NotImplementedError("return_features is not available together with lengths")
            lens = _lengths_tensor(lengths, B)
            if B > 0 and T > 0:
                _native.check(eng.lib.vasr_forward_ragged(eng.handle, _native.ptr(mel), _native.ptr(lens), B, T,
                                                          _native.ptr(logits), _stream_ptr(mel.device)))
            return back(logits)
        feats = None
        if return_features:
            feats = {k: torch.empty(B, L, self.config.d_model, device=mel.device, dtype=torch.float32)
                     for k in ("temporal_binding", "local_features", "fused_features")}
        if B > 0 and T > 0:
            _native.check(eng.lib.vasr_forward(
                eng.handle, _native.ptr(mel), B, T, _native.ptr(logits),
                _native.ptr(feats["temporal_binding"]) if feats else None,
                _native.ptr(feats["local_features"]) if feats else None,
                _native.ptr(feats["fused_features"]) if feats else None, _stream_ptr(mel.device)))
        if return_features:
            return back(logits), {k: back(v) for k, v in feats.items()}
        return back(logits)

    def get_output_length(self, input_length: int) -> int:
        """model.py:370-383"""
        return (input_length + 1) // 2

    @torch.no_grad()
    def transcribe(self, audio: torch.Tensor, lengths=None) -> List[List[int]]:
        """Fused fast path: 16 kHz PCM (S,) | (B, S) -> greedy CTC token ids per utterance
        (compute_mel_spectrogram -> forward -> ctc_greedy_decode, scripts/transcribe.py:69-82).
        A CUDA tensor is consumed in place; a CPU tensor is copied host->device inside the call
        (pin it for full PCIe speed) and only the token ids come back.
        `lengths` (B sample counts): a ragged batch padded to S; utterance b is its first lengths[b] samples
        and is transcribed exactly as transcribe(audio[b, :lengths[b]]) would (own reflect padding, mel
        statistics, pooling windows, attention keys and decode length) in the same launches as its mates."""
        if audio.dim() == 1:
            audio = audio.unsqueeze(0)
        B, S = audio.shape
        dev = self._exec_device(audio)
        eng = self._engine(dev)
        L = self.get_output_length(1 + S // 160)
        slen = None if lengths is None else _lengths_tensor(lengths, B)
        if audio.device.type == "cpu":
            pcm = audio.to(torch.float32).contiguous()
            # pinned result buffers are kept per shape: a cudaHostAlloc per call costs more than the D2H itself
            # (the lists returned below are copies)
            cache = self.__dict__.setdefault("_pinned_out", {})
            if (B, L) not in cache:
                if len(cache) >= 8:
                    cache.clear()
                cache[(B, L)] = (torch.empty(B, L, dtype=torch.int32, pin_memory=True),
                                 torch.empty(B, dtype=torch.int32, pin_memory=True))
            tokens, lens = cache[(B, L)]
            if slen is None:
                _native.check(eng.lib.vasr_transcribe_host(eng.handle, _native.ptr(pcm), B, S, _native.ptr(tokens),
                                                           _native.ptr(lens)))
            else:
                _native.check(eng.lib.vasr_transcribe_ragged_host(eng.handle, _native.ptr(pcm), _native.ptr(slen), B, S,
                                                                  _native.ptr(tokens), _native.ptr(lens)))
            return _token_lists(tokens, lens)
        else:
            pcm = self._check_input(audio, "audio")
            tokens = torch.empty(B, L, dtype=torch.int32, device=pcm.device)
            lens = torch.empty(B, dtype=torch.int32, device=pcm.device)
            if slen is None:
                _native.check(eng.lib.vasr_transcribe(eng.handle, _native.ptr(pcm), B, S, _native.ptr(tokens),
                                                      _native.ptr(lens), _stream_ptr(pcm.device)))
            else:
                _native.check(eng.lib.vasr_transcribe_ragged(eng.handle, _native.ptr(pcm), _native.ptr(slen), B, S,
                                                             _native.ptr(tokens), _native.ptr(lens),
                                                             _stream_ptr(pcm.device)))
            tokens, lens = tokens.cpu(), lens.cpu()
        return _token_lists(tokens, lens)

    @torch.no_grad()
    def transcribe_beam(self, audio: torch.Tensor, lengths=None, beam_width: int = 10, lm_scorer=None,
                        lm_weight: float = 0.0, word_score: float = 0.0):
        """Fused PCM -> n-best: 16 kHz PCM (S,) | (B, S) -> per utterance its `beam_width` best prefixes
        (List[List[DecodingResult]], best first, text ""), in one native call: log-mel, forward, the CTC head writing
        logits, and the device prefix beam search (ctc_beam_search, blank 0), with or without an NGramLM /
        WordNGramLM under the same rules and errors.  The LM must live on the model's execution device.
        `lengths` (B sample counts): a ragged batch as in transcribe().  Utterance b gets bit for bit
        ctc_beam_search(forward(compute_mel_spectrogram(audio[b, :lengths[b]]).unsqueeze(0)), ...)[0].
        A CUDA tensor is consumed in place; a CPU tensor (pin it) is copied in inside the call."""
        from .decode import _beam_results, _check_lm_fits, _search_lm
        lm = _search_lm(lm_scorer, lm_weight, word_score)
        if audio.dim() == 1:
            audio = audio.unsqueeze(0)
        B, S = audio.shape
        dev = self._exec_device(audio)
        slen = None if lengths is None else _lengths_tensor(lengths, B)
        if lm is not None:
            _check_lm_fits(lm, self.config.vocab_size, 0)
            if lm.device.index != (dev.index if dev.index is not None else torch.cuda.current_device()):
                raise ValueError(f"the LM is on {lm.device}, the model runs on {dev}")
        W = int(beam_width)
        if not 1 <= W <= 32:       # before the result buffers are sized by it; the library's rule and exception type
            raise ValueError(f"beam_width must be in [1, 32], got {W}")
        eng = self._engine(dev)
        L = self.get_output_length(1 + S // 160)
        hlm = lm._handle if lm is not None else None
        if audio.device.type == "cpu":
            pcm = audio.to(torch.float32).contiguous()
            cache = self.__dict__.setdefault("_pinned_beam_out", {})   # per shape, as transcribe() does
            if (B, W, L) not in cache:
                if len(cache) >= 8:
                    cache.clear()
                cache[(B, W, L)] = (torch.empty(B, W, L, dtype=torch.int32, pin_memory=True),
                                    torch.empty(B, W, dtype=torch.int32, pin_memory=True),
                                    torch.empty(B, W, dtype=torch.float64, pin_memory=True))
            tokens, lens, scores = cache[(B, W, L)]
            _native.check(eng.lib.vasr_transcribe_beam_host(
                eng.handle, _native.ptr(pcm), _native.ptr(slen), B, S, W, hlm, float(lm_weight), float(word_score),
                _native.ptr(tokens), _native.ptr(lens), _native.ptr(scores)))
        else:
            pcm = self._check_input(audio, "audio")
            tokens = torch.empty(B, W, L, dtype=torch.int32, device=pcm.device)
            lens = torch.empty(B, W, dtype=torch.int32, device=pcm.device)
            scores = torch.empty(B, W, dtype=torch.float64, device=pcm.device)
            _native.check(eng.lib.vasr_transcribe_beam(
                eng.handle, _native.ptr(pcm), _native.ptr(slen), B, S, W, hlm, float(lm_weight), float(word_score),
                _native.ptr(tokens), _native.ptr(lens), _native.ptr(scores), _stream_ptr(pcm.device)))
        return _beam_results(tokens, lens, scores)

    @torch.no_grad()
    def align(self, audio: torch.Tensor, targets: List[List[int]], lengths=None):
        """Fused PCM -> forced alignment: 16 kHz PCM (S,) | (B, S) and one target (token ids) per utterance -> per
        utterance an AlignmentResult (ctc_forced_align's, blank 0), in one native call: log-mel, forward, the CTC head
        writing logits, and the device Viterbi alignment.  `lengths` (B sample counts): a ragged batch as in
        transcribe().  Utterance b gets bit for bit ctc_forced_align(forward(compute_mel_spectrogram(
        audio[b, :lengths[b]]).unsqueeze(0)), targets[b:b+1])[0].  Host PCM is staged to the execution device."""
        from .decode import _align_targets, _alignment_results
        if audio.dim() == 1:
            audio = audio.unsqueeze(0)
        B, S = audio.shape
        tgt, tlens, U_max = _align_targets(targets, B, self.config.vocab_size, 0)
        slen = None if lengths is None else _lengths_tensor(lengths, B)
        dev = self._exec_device(audio)
        eng = self._engine(dev)
        pcm = self._check_input(audio, "audio")
        L = self.get_output_length(1 + S // 160)
        labels = torch.empty(B, L, dtype=torch.int32, device=pcm.device)
        lps = torch.empty(B, L, dtype=torch.float32, device=pcm.device)
        scores = torch.empty(B, dtype=torch.float64, device=pcm.device)
        _native.check(eng.lib.vasr_align(eng.handle, _native.ptr(pcm), _native.ptr(slen), B, S, _native.ptr(tgt),
                                         _native.ptr(tlens), U_max, _native.ptr(labels), _native.ptr(lps),
                                         _native.ptr(scores), _stream_ptr(pcm.device)))
        frames = [L] * B if slen is None else [self.get_output_length(1 + n // 160) for n in slen.tolist()]
        return _alignment_results(tgt, tlens, labels, lps, scores, frames, 0)

    @torch.no_grad()
    def transcribe_batches(self, batches: Iterable[torch.Tensor], as_arrays: bool = False
                           ) -> Iterator[List[List[int]]]:
        """transcribe() over a stream of host batches, pipelined: while the kernels of batch i run,
        batch i+1 is copied host->device on a second stream and the token ids of batch i-1 are copied
        back and turned into lists.  Yields one List[List[int]] per input batch, in order; results
        are identical to calling transcribe() on each batch.  Batches are (B, S) float32 CPU
        tensors (pin them for full PCIe speed); shapes may change from batch to batch.  An item may also
        be a pair (batch, lengths): a ragged batch, as transcribe(batch, lengths=lengths).  The input iterator is
        read one batch ahead of the batch being computed.
        as_arrays=True yields (tokens (B, L) int32 left-packed, counts (B,) int32) numpy copies instead of lists:
        the compact form sharding.gather_token_arrays exchanges between ranks."""
        dev = self._exec_device()
        eng = self._engine(dev)
        comp = torch.cuda.current_stream(dev)
        copy = torch.cuda.Stream(dev)
        back = torch.cuda.Stream(dev)
        # three device slots: the batch whose kernels run, the next one (its host->device copy is issued as soon as
        # the current batch's kernels are queued, i.e. a whole step ahead of its use: with 8 ranks sharing the host's
        # PCIe and memory a 61 MB copy takes several ms) and the previous one (results not yet collected)
        slots = [dict(pcm=None, tok=None, lens=None, tok_h=None, lens_h=None, shape=None, slen=None,
                      h2d=torch.cuda.Event(), done=torch.cuda.Event(), free=torch.cuda.Event()) for _ in range(3)]

        def stage(audio, sl):
            slen = None
            if isinstance(audio, (tuple, list)):        # (padded batch, per-utterance sample counts): ragged
                audio, slen = audio
            if audio.device.type != "cpu":
                raise RuntimeError("transcribe_batches takes host batches; use transcribe() for CUDA tensors")
            if audio.dim() == 1:
                audio = audio.unsqueeze(0)
            audio = audio.to(torch.float32).contiguous()
            B, S = audio.shape
            L = self.get_output_length(1 + S // 160)
            if sl["pcm"] is None or sl["pcm"].shape != (B, S):
                sl["pcm"] = torch.empty(B, S, device=dev, dtype=torch.float32)
                sl["tok"] = torch.empty(B, L, device=dev, dtype=torch.int32)
                sl["lens"] = torch.empty(B, device=dev, dtype=torch.int32)
                sl["tok_h"] = torch.empty(B, L, dtype=torch.int32, pin_memory=True)
                sl["lens_h"] = torch.empty(B, dtype=torch.int32, pin_memory=True)
                copy.wait_stream(comp)          # a re-allocated buffer may still be in use by queued kernels
            with torch.cuda.stream(copy):
                copy.wait_event(sl["free"])      # the kernels that last read this slot's PCM are done
                sl["pcm"].copy_(audio, non_blocking=True)
                sl["h2d"].record(copy)
            sl["shape"], sl["slen"] = (B, S), slen
            sl["src"] = audio                    # keeps a converted copy alive until the transfer has been consumed
            return sl

        it = iter(batches)
        first = next(it, None)
        staged = stage(first, slots[0]) if first is not None else None
        pending = None          # slot of the batch whose results are still on the device
        i = 0
        while staged is not None:
            sl = staged
            B, S = sl["shape"]
            comp.wait_event(sl["h2d"])
            comp.wait_event(sl["done"])          # the slot's previous results have left the device buffers
            if sl["slen"] is None:
                _native.check(eng.lib.vasr_transcribe(eng.handle, _native.ptr(sl["pcm"]), B, S, _native.ptr(sl["tok"]),
                                                      _native.ptr(sl["lens"]), ctypes.c_void_p(comp.cuda_stream)))
            else:
                slen_t = _lengths_tensor(sl["slen"], B)  # stays referenced across the call (read synchronously)
                _native.check(eng.lib.vasr_transcribe_ragged(
                    eng.handle, _native.ptr(sl["pcm"]), _native.ptr(slen_t), B, S,
                    _native.ptr(sl["tok"]), _native.ptr(sl["lens"]), ctypes.c_void_p(comp.cuda_stream)))
            sl["free"].record(comp)
            # results travel on a stream of their own: on the compute stream the two small D2H copies would sit
            # between this batch's last kernel and the next batch's first
            with torch.cuda.stream(back):
                back.wait_event(sl["free"])
                sl["tok_h"].copy_(sl["tok"], non_blocking=True)
                sl["lens_h"].copy_(sl["lens"], non_blocking=True)
                sl["done"].record(back)
            i += 1
            nxt = next(it, None)
            staged = stage(nxt, slots[i % 3]) if nxt is not None else None
            if pending is not None:
                yield self._collect(pending, as_arrays)
            pending = sl
        if pending is not None:
            yield self._collect(pending, as_arrays)

    @staticmethod
    def _collect(sl, as_arrays: bool = False):
        sl["done"].synchronize()
        if as_arrays:
            return sl["tok_h"].numpy().copy(), sl["lens_h"].numpy().copy()
        return _token_lists(sl["tok_h"], sl["lens_h"])

    @torch.no_grad()
    def transcribe_list(self, utterances: List[torch.Tensor], max_batch: int = 64) -> List[List[int]]:
        """Variable-length input: a list of 1-D PCM tensors -> token ids per utterance, in input order.
        The reference's collator pads with zeros and never masks (data.py:145-203), which makes an
        utterance's result depend on its batch mates.  Here the utterances are sorted by length, cut into
        batches of at most `max_batch`, padded to the longest of the batch and run as ragged batches
        (transcribe(..., lengths=...)), so every result equals transcribe() of that utterance alone."""
        out: List[Optional[List[int]]] = [None] * len(utterances)
        for u in utterances:
            if u.dim() != 1:
                raise RuntimeError("transcribe_list takes 1-D PCM tensors")
        order = sorted(range(len(utterances)), key=lambda i: int(utterances[i].numel()))
        dev = self._exec_device()
        for j in range(0, len(order), max_batch):
            part = order[j:j + max_batch]
            lens = [int(utterances[i].numel()) for i in part]
            batch = torch.zeros(len(part), max(lens), device=dev, dtype=torch.float32)
            for r, i in enumerate(part):
                batch[r, :lens[r]] = utterances[i].to(dev, torch.float32)
            for i, toks in zip(part, self.transcribe(batch, lengths=lens)):
                out[i] = toks
        return out  # type: ignore[return-value]

    def extend_positional_table(self, rows: int) -> None:
        """Regenerate pe_time with `rows` rows by the formula of model.py:94-100.  The reference
        stops at 5000 tokens (~100 s) and raises beyond; long-form input needs a longer table."""
        pos = self.temporal_binding.pos_encoding
        pos.pe_time = time_table(rows, self.config.d_model).to(pos.pe_time.device)

    @classmethod
    def from_pretrained(cls, model_name_or_path: str, quantized: bool = False, **kwargs) -> "VELOCITYASR":
        """model.py:385-433: local checkpoint with keys 'config' and 'model_state_dict' (or a bare
        state dict).  Hub names are not implemented in the reference either."""
        if not os.path.exists(model_name_or_path):
            raise NotImplementedError(
                "Model hub download not yet implemented. Please provide a local path to the checkpoint.")
        ckpt = torch.load(model_name_or_path, map_location="cpu")
        # save_pretrained files carry the model config under 'config' (model.py:455-460); Trainer
        # checkpoints carry the TRAINING config there and the model's under 'model_config'
        # (training.py:382-397) — the reference reads the wrong one and silently falls back to defaults
        # (SURVEY.md 5.4); prefer 'model_config' when it is present.
        if "model_config" in ckpt:
            cfg = VelocityASRConfig.from_dict(dict(ckpt["model_config"]))
        elif "config" in ckpt:
            cfg = VelocityASRConfig.from_dict(dict(ckpt["config"]))
        else:
            cfg = VelocityASRConfig()
        model = cls(cfg)
        sd = ckpt["model_state_dict"] if "model_state_dict" in ckpt else ckpt
        rows = sd["temporal_binding.pos_encoding.pe_time"].shape[0]
        if rows != 5000:
            model.extend_positional_table(rows)
        model.load_state_dict(sd)
        return model

    def save_pretrained(self, save_path: str):
        """model.py:435-467"""
        os.makedirs(os.path.dirname(save_path) or ".", exist_ok=True)
        torch.save({"config": self.config.to_dict(), "model_state_dict": self.state_dict()}, save_path)

    def count_parameters(self) -> int:
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    # ---- module-level seams for parity tests (reference classes SSMBlock, HierarchicalGlobalContext,
    # CTCOutputHead) ----------------------------------------------------------------------------
    @torch.no_grad()
    def run_ssm_block(self, x: torch.Tensor, layer: int, stack: str = "local", scan_mode: Optional[str] = None):
        x = self._check_input(x, "x")
        eng = self._engine(x.device)
        out = torch.empty_like(x)
        mode = -1 if scan_mode is None else _native.SCAN_MODE_ID[scan_mode]
        _native.check(eng.lib.vasr_ssm_block(eng.handle, 0 if stack == "local" else 1, layer, mode, _native.ptr(x),
                                             x.size(0), x.size(1), _native.ptr(out), _stream_ptr(x.device)))
        return out

    @torch.no_grad()
    def run_global_context(self, local_features: torch.Tensor):
        x = self._check_input(local_features, "local_features")
        eng = self._engine(x.device)
        out = torch.empty_like(x)
        _native.check(eng.lib.vasr_global_context(eng.handle, _native.ptr(x), x.size(0), x.size(1), _native.ptr(out),
                                                  _stream_ptr(x.device)))
        return out

    @torch.no_grad()
    def run_ctc_head(self, x: torch.Tensor):
        x = self._check_input(x, "x")
        eng = self._engine(x.device)
        out = torch.empty(x.size(0), x.size(1), self.config.vocab_size, device=x.device, dtype=torch.float32)
        _native.check(eng.lib.vasr_ctc_head(eng.handle, _native.ptr(x), x.size(0), x.size(1), _native.ptr(out),
                                            _stream_ptr(x.device)))
        return out
