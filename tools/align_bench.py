"""Time CTC forced alignment and transcript log-likelihood on the device at the beam search's headline shape
(64 x 751 frames x vocab 1000), and the fused PCM -> alignment path.

    python tools/align_bench.py [--batch 64] [--frames 751] [--vocab 1000] [--reps 15] [--out FILE]

Seeded logits (seed 0, as tools/beam_bench.py) and seeded targets of about L/3 and L/2 tokens, over the full frames
and over a ragged batch (lengths uniform in [L/4, L], targets scaled to each length).  For each: ctc_forced_align
and ctc_log_likelihood (Python calls, host results included), median and fastest of individually synchronised calls
(the GPU may be shared, and one delayed call would dominate a mean); the native entry points alone; the LM-free beam
search (W = 10) on the same logits, for comparison.  Then VELOCITYASR.align on 64 x 15 s PCM (seed 1234,
random-init weights, sequential scan) against mel + forward + ctc_forced_align called separately, and the same
utterances through torchaudio's CPU forced_align one at a time, for scale.  The card's name and power limit are
read in the same run and stored with the results.  --out FILE also writes the JSON to FILE.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "velocity-asr_b200"))
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
import velocity_asr as va  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--frames", type=int, default=751)
ap.add_argument("--vocab", type=int, default=1000)
ap.add_argument("--reps", type=int, default=15)
ap.add_argument("--out", default="", help="also write the JSON result to this file")
a = ap.parse_args()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power = (s.strip() for s in q.stdout.strip().split(","))
        return name, power
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def timed_fn(fn, n=a.reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    fastest[0] = min(ts)
    return statistics.median(ts), res


fastest = [0.0]   # the fastest call of the last timed_fn: on a shared GPU the least disturbed one


def rec(key, dt):
    """Store the median and the fastest call of the last timed_fn under key."""
    out[key + "_ms"] = round(dt * 1e3, 3)
    out[key + "_fastest_ms"] = round(fastest[0] * 1e3, 3)


def targets_for(rs, lens, frac, V):
    """Per utterance about frac * its frames tokens, ids in [1, V), no two equal neighbours (so every target fits)."""
    out = []
    for n in lens:
        U = max(int(n * frac), 0)
        y = rs.randint(1, V, size=U)
        for i in range(1, U):
            if y[i] == y[i - 1]:
                y[i] = y[i] % (V - 1) + 1
        out.append(y.tolist())
    return out


assert torch.cuda.is_available(), "align_bench needs a CUDA device"
B, L, V = a.batch, a.frames, a.vocab
g = torch.Generator(device="cuda").manual_seed(0)
lg = torch.randn(B, L, V, device="cuda", generator=g) * 3.0
name, power = card()
out = {"what": "CTC forced alignment / log-likelihood on the device: Python calls with host results (native_*: the C "
               f"entry point alone), median and fastest of {a.reps} individually synchronised calls",
       "gpu": name, "power_limit": power,
       "batch": B, "frames": L, "vocab": V}
rs = np.random.RandomState(0)
ragged_lens = torch.randint(L // 4, L + 1, (B,), generator=torch.Generator().manual_seed(1)).tolist()
out["ragged_lengths_min_mean_max"] = [min(ragged_lens), round(sum(ragged_lens) / B, 1), max(ragged_lens)]
for tag, frac in (("u_third", 1 / 3), ("u_half", 1 / 2)):
    for rtag, lens in (("full", None), ("ragged", ragged_lens)):
        tg = targets_for(rs, [L] * B if lens is None else lens, frac, V)
        dt_a, res = timed_fn(lambda: va.ctc_forced_align(lg, tg, lengths=lens))
        rec(f"align_{tag}_{rtag}", dt_a)
        dt_l, ll = timed_fn(lambda: va.ctc_log_likelihood(lg, tg, lengths=lens))
        rec(f"log_likelihood_{tag}_{rtag}", dt_l)
        out.update({f"tokens_{tag}_{rtag}_mean": round(sum(map(len, tg)) / B, 1),
                    f"all_fit_{tag}_{rtag}": all(r.timestamps is not None for r in res)})
        if tag == "u_third" and rtag == "full":
            lp = torch.log_softmax(lg, -1).cpu()
            fa = torch.from_numpy(np.ascontiguousarray(lp.numpy()))
            ta_tg = [torch.tensor([y], dtype=torch.int32) for y in tg]

            def torchaudio_loop():
                import torchaudio.functional as F
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    return [F.forced_align(fa[b:b + 1], ta_tg[b], blank=0)[0] for b in range(B)]
            try:
                t0 = time.perf_counter()
                ta = torchaudio_loop()
                dt_t = time.perf_counter() - t0
                t0 = time.perf_counter()
                torchaudio_loop()
                dt_t = min(dt_t, time.perf_counter() - t0)
                out.update({"torchaudio_cpu_forced_align_u_third_full_ms": round(dt_t * 1e3, 3),
                            "torchaudio_cpu_threads": torch.get_num_threads(),
                            "torchaudio_same_paths": sum(int(ta[b][0].tolist() == res[b].frame_labels.tolist())
                                                         for b in range(B))})
            except ImportError:
                out["torchaudio_cpu_forced_align_u_third_full_ms"] = "not measured: no torchaudio"


# the native entry points alone (argument checks, scratch, row statistics, kernel; no host result lists), u_third
# over the full frames, and the LM-free beam search (W = 10) on the same logits for comparison
from velocity_asr import _native  # noqa: E402
from velocity_asr.decode import _align_targets  # noqa: E402
tg = targets_for(np.random.RandomState(0), [L] * B, 1 / 3, V)
tgt, tlens, U_max = _align_targets(tg, B, V, 0)
labels = torch.empty(B, L, dtype=torch.int32, device="cuda")
lps = torch.empty(B, L, dtype=torch.float32, device="cuda")
scores = torch.empty(B, dtype=torch.float64, device="cuda")
stream = lambda: __import__("ctypes").c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
lib = _native.lib()
rec("native_align_u_third_full", timed_fn(lambda: _native.check(lib.vasr_ctc_align(
    _native.ptr(lg), None, B, L, V, 0, 0, _native.ptr(tgt), _native.ptr(tlens), U_max, _native.ptr(labels),
    _native.ptr(lps), _native.ptr(scores), stream())))[0])
rec("native_log_likelihood_u_third_full", timed_fn(lambda: _native.check(lib.vasr_ctc_log_likelihood(
    _native.ptr(lg), None, B, L, V, 0, 0, _native.ptr(tgt), _native.ptr(tlens), U_max, _native.ptr(scores),
    stream())))[0])
rec("beam_search_w10_same_logits", timed_fn(lambda: va.ctc_beam_search(lg, beam_width=10))[0])

import fixtures_util as FU  # noqa: E402
torch.manual_seed(0)
model = va.VELOCITYASR(va.VelocityASRConfig(scan_mode="sequential")).cuda().eval()
pcm = FU.synth_audio(64, 16000 * 15, seed=1234).cuda()
Lp = model.get_output_length(1 + pcm.shape[1] // 160)
ptg = targets_for(rs, [Lp] * 64, 1 / 3, model.config.vocab_size)


def composed():
    return va.ctc_forced_align(model(va.compute_mel_spectrogram(pcm)), ptg)


def fields(res):
    return [(r.frame_labels.tolist(), r.score) for r in res]


out["pcm"] = "64 x 15 s PCM (seed 1234), random-init weights, scan_mode=sequential, targets of L/3 tokens"
dt_f, res_f = timed_fn(lambda: model.align(pcm, ptg))
rec("model_align", dt_f)
dt_c, res_c = timed_fn(composed)
rec("mel_forward_plus_align", dt_c)
rec("mel_forward", timed_fn(lambda: model(va.compute_mel_spectrogram(pcm)))[0])
out["model_align_equals_composed"] = fields(res_f) == fields(res_c)
print(json.dumps(out))
if a.out:
    with open(a.out, "w") as f:
        f.write(json.dumps(out, indent=1) + "\n")
