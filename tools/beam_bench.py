"""Time the device prefix beam search at the headline shape (64 x 751 frames x vocab 1000, width 10).

    python tools/beam_bench.py [--width 10] [--batch 64] [--lm-order N] [--word-lm-order N]

--lm-order N also writes a seeded synthetic order-N ARPA LM (tests/lm_oracle.py) to a temporary file, loads
it, and times the LM-free and the LM-fused search in the same process on the same logits.
--word-lm-order N does the same with a synthetic order-N word-level LM (tests/word_lm_oracle.py) and times the
word-fused search, lexicon-free and lexicon-constrained.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "velocity-asr_b200"))
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
sys.path.insert(0, os.path.join(HERE, "..", "oracle"))
import velocity_asr as va  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--width", type=int, default=10)
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--frames", type=int, default=751)
ap.add_argument("--vocab", type=int, default=1000)
ap.add_argument("--lm-order", type=int, default=0, help="also time the search fused with an order-N n-gram LM")
ap.add_argument("--lm-ngrams", type=int, default=100000, help="n-grams per order above 1 in the synthetic LM")
ap.add_argument("--lm-weight", type=float, default=0.5)
ap.add_argument("--word-lm-order", type=int, default=0, help="also time the search fused with an order-N word LM")
ap.add_argument("--word-lm-words", type=int, default=20000, help="words in the synthetic word LM")
ap.add_argument("--word-score", type=float, default=0.5)
a = ap.parse_args()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power = (s.strip() for s in q.stdout.strip().split(","))
        return name, power
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def timed(**kw):
    for _ in range(2):
        va.ctc_beam_search(lg, beam_width=a.width, **kw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = 5
    for _ in range(n):
        res = va.ctc_beam_search(lg, beam_width=a.width, **kw)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n, res


g = torch.Generator(device="cuda").manual_seed(0)
lg = torch.randn(a.batch, a.frames, a.vocab, device="cuda", generator=g) * 3.0
name, power = card()
out = {"what": "ctc_beam_search on the device, host result lists included", "gpu": name, "power_limit": power,
       "batch": a.batch, "frames": a.frames, "vocab": a.vocab, "beam_width": a.width}
dt, res = timed()
out.update({"ms_per_batch": round(dt * 1e3, 3), "best_beam_len": len(res[0][0].tokens)})
if a.lm_order > 0:
    import lm_oracle as LO
    vocab = va.create_default_vocabulary(a.vocab)[:a.vocab]
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "synthetic.arpa")
        ngrams = LO.write_synthetic_arpa(path, vocab, order=a.lm_order, seed=0, per_order=a.lm_ngrams)
        t0 = time.perf_counter()
        lm = va.NGramLM.from_arpa(path, vocab)
        load = time.perf_counter() - t0
    dt_lm, res_lm = timed(lm_scorer=lm, lm_weight=a.lm_weight)
    out.update({"lm_order": a.lm_order, "lm_ngrams": ngrams, "lm_weight": a.lm_weight,
                "lm_load_s": round(load, 3), "lm_ms_per_batch": round(dt_lm * 1e3, 3),
                "lm_over_lm_free": round(dt_lm / dt, 2), "lm_best_beam_len": len(res_lm[0][0].tokens)})
    lm.close()
if a.word_lm_order > 0:
    import string
    import word_lm_oracle as WO
    vocab = va.create_default_vocabulary(a.vocab)[:a.vocab]
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "synthetic_words.arpa")
        WO.write_synthetic_word_arpa(path, string.ascii_lowercase, order=a.word_lm_order, seed=0,
                                     n_words=a.word_lm_words, per_order=a.lm_ngrams)
        t0 = time.perf_counter()
        wlm = va.WordNGramLM.from_arpa(path, vocab)
        load = time.perf_counter() - t0
        clm = va.WordNGramLM.from_arpa(path, vocab, lexicon_constrained=True)
    out.update({"word_lm_order": a.word_lm_order, "word_lm_lexicon": wlm.lexicon_size, "word_lm_load_s": round(load, 3),
                "word_lm_weight": a.lm_weight, "word_score": a.word_score})
    for tag, m in (("word_lm", wlm), ("word_lm_constrained", clm)):
        dt_w, res_w = timed(lm_scorer=m, lm_weight=a.lm_weight, word_score=a.word_score)
        out.update({f"{tag}_ms_per_batch": round(dt_w * 1e3, 3), f"{tag}_over_lm_free": round(dt_w / dt, 2),
                    f"{tag}_best_beam_len": len(res_w[0][0].tokens) if res_w[0] else -1})
        m.close()
print(json.dumps(out))
