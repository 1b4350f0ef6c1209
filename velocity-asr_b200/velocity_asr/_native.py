"""ctypes binding of libvasr.so (include/vasr.h).  There is no fallback: if the library is
missing, or there is no CUDA device, every compute entry point raises."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VASR_LIB") or os.path.join(_HERE, "libvasr.so")   # VASR_LIB: A/B runs of two builds

OK, ERR_INVALID, ERR_SHAPE, ERR_CUDA, ERR_STATE, ERR_UNSUPPORTED = range(6)
SCAN_MODE_ID = {"sequential": 0, "parallel": 1, "mamba": 2}


class VasrConfig(ctypes.Structure):
    _fields_ = [(n, c_int32) for n in (
        "mel_bins", "d_model", "ssm_layers", "ssm_state_dim", "ssm_expand_ratio", "ssm_kernel_size",
        "global_ssm_layers", "global_ssm_state_dim", "attention_heads", "attention_dim", "vocab_size",
        "scan_mode")]


_SIGNATURES = {
    "vasr_last_error": (c_char_p, []),
    "vasr_version": (c_char_p, []),
    "vasr_create": (c_int, [POINTER(VasrConfig), c_int, POINTER(c_void_p)]),
    "vasr_destroy": (None, [c_void_p]),
    "vasr_set_weight": (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    "vasr_commit_weights": (c_int, [c_void_p]),
    "vasr_num_frames": (c_int64, [c_int64]),
    "vasr_num_tokens": (c_int64, [c_int64]),
    "vasr_log_mel": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "vasr_forward": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_ssm_block": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "vasr_global_context": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "vasr_ctc_head": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "vasr_selective_scan": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                    c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64,
                                    c_int64, c_int64, c_int, c_void_p]),
    "vasr_ctc_greedy": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "vasr_ctc_greedy_timestamps": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p]),
    "vasr_ctc_greedy_confidence": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe_timestamps": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe_timestamps_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_ctc_beam_search": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                     c_void_p]),
    "vasr_lm_create_arpa": (c_int, [c_char_p, c_void_p, c_int64, c_int, c_int, POINTER(c_void_p)]),
    "vasr_lm_destroy": (None, [c_void_p]),
    "vasr_lm_order": (c_int, [c_void_p]),
    "vasr_lm_log_prob": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "vasr_ctc_beam_search_lm": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_double,
                                        c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_lm_create_word_arpa": (c_int, [c_char_p, c_void_p, c_int64, c_int, c_char_p, c_int, c_int, POINTER(c_void_p)]),
    "vasr_lm_word_ids": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "vasr_lm_lexicon_size": (c_int64, [c_void_p]),
    "vasr_ctc_beam_search_word_lm": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_double,
                                             c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_ctc_beam_search_ragged": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p,
                                            c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe_beam": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_double,
                                     c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe_beam_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_double,
                                          c_double, c_void_p, c_void_p, c_void_p]),
    "vasr_ctc_align": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p,
                               c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "vasr_ctc_log_likelihood": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p,
                                        c_void_p, c_int64, c_void_p, c_void_p]),
    "vasr_align": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                           c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe_host": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "vasr_transcribe_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "vasr_transcribe_ragged_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "vasr_forward_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "vasr_linear": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64,
                            c_int, c_void_p]),
    "vasr_set_quantization": (c_int, [c_void_p, c_int]),
    "vasr_calibrate": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "vasr_get_quant_params": (c_int, [c_void_p, c_char_p, POINTER(c_float), POINTER(c_float)]),
    "vasr_set_quant_params": (c_int, [c_void_p, c_char_p, c_float, c_float]),
    "vasr_quant_site": (c_int, [c_void_p, c_char_p, c_void_p, c_int64, c_int64, c_void_p, POINTER(c_int32),
                                POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "vasr_split_tf32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "vasr_linear_tc": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                               c_int64, c_int64, c_int64, c_int, c_void_p]),
    "vasr_kernel_launches": (c_int64, [c_void_p]),
    "vasr_tc_launches": (c_int64, [c_void_p]),
    "vasr_workspace_bytes": (c_int64, [c_void_p]),
    "vasr_set_timing": (c_int, [c_void_p, c_int]),
    "vasr_last_timing": (c_int, [c_void_p, POINTER(c_float), POINTER(c_int32), POINTER(c_float)]),
}

_lib = None


def lib():
    """Load libvasr.so once.  Loading needs no GPU; calling compute entry points does."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python velocity-asr_b200/build.py` "
                "(or __graft_entry__.build()).  There is no CPU or PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


_EXC = {ERR_INVALID: ValueError, ERR_SHAPE: RuntimeError, ERR_CUDA: RuntimeError, ERR_STATE: RuntimeError,
        ERR_UNSUPPORTED: NotImplementedError}


def check(code: int):
    """Map a C status to the exception type the reference raises for the same condition
    (ValueError for an unknown scan_mode, ssm.py:126; RuntimeError for a shape the model cannot
    take, model.py:125; NotImplementedError for unsupported configurations)."""
    if code != OK:
        msg = lib().vasr_last_error().decode("utf-8", "replace")
        raise _EXC.get(code, RuntimeError)(f"libvasr: {msg}")


def default_cuda_device():
    """The CUDA device host-resident inputs are staged to when neither the input nor the model names one
    (the process's current device).  Raises when there is none: this build has no CPU path."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("velocity_asr (B200 build): no CUDA device is available and there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def ptr(t):
    """Device (or host) address of a contiguous float32/int32 tensor, or None."""
    return None if t is None else c_void_p(t.data_ptr())
