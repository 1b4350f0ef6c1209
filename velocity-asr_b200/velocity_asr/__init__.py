"""velocity_asr — B200-native drop-in for the inference path of shaderko/velocity-asr.

Same import name and the same callables as the reference package for the hot path
(velocity_asr/__init__.py:95-145): VelocityASRConfig, VELOCITYASR, from_pretrained,
compute_mel_spectrogram, ctc_greedy_decode, CTCDecoder, create_default_vocabulary — plus
config_from_yaml (the mapping the reference keeps in scripts/train.py:158-174), the fused
VELOCITYASR.transcribe, and the scan operator.  All arithmetic runs in libvasr.so
(hand-written sm_100a CUDA behind the C ABI of include/vasr.h); there is no CPU fallback.
"""
__version__ = "2.0.0+b200"

from .config import VelocityASRConfig, config_from_yaml, SCAN_MODES
from .model import VELOCITYASR
from .audio import compute_mel_spectrogram, SAMPLE_RATE, N_FFT, HOP_LENGTH, N_MELS
from .decode import (ctc_greedy_decode, ctc_greedy_decode_with_timestamps, ctc_beam_search, DecodingResult, CTCDecoder,
                  ctc_forced_align, ctc_log_likelihood, AlignmentResult,
                  create_default_vocabulary, frames_to_seconds, words_with_timestamps,
                  BLANK_TOKEN)
from .lm import NGramLM, WordNGramLM
from .ops import selective_scan, selective_scan_fn, linear, split_tf32
from .quantize import QuantizationConfig, prepare_model_for_qat, calibrate_model

MAMBA_AVAILABLE = True  # scan_mode="mamba" is served by the in-tree scan kernel (ssm.py:20-26)


def from_pretrained(model_name_or_path: str, **kwargs) -> VELOCITYASR:
    """velocity_asr/__init__.py:82-92"""
    return VELOCITYASR.from_pretrained(model_name_or_path, **kwargs)


__all__ = [
    "__version__", "VELOCITYASR", "VelocityASRConfig", "config_from_yaml", "from_pretrained",
    "compute_mel_spectrogram", "SAMPLE_RATE", "N_FFT", "HOP_LENGTH", "N_MELS",
    "ctc_greedy_decode", "ctc_greedy_decode_with_timestamps", "ctc_beam_search", "DecodingResult", "CTCDecoder", "create_default_vocabulary", "BLANK_TOKEN",
    "ctc_forced_align", "ctc_log_likelihood", "AlignmentResult",
    "NGramLM", "WordNGramLM",
    "frames_to_seconds", "words_with_timestamps",
    "selective_scan", "selective_scan_fn", "linear", "split_tf32", "MAMBA_AVAILABLE", "SCAN_MODES",
    "QuantizationConfig", "prepare_model_for_qat", "calibrate_model",
]
