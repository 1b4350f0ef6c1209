"""Time the greedy transcript with token timestamps and scores at config 2 (64 x 15 s PCM, default model).

    python tools/timestamps_bench.py [--reps 15] [--rounds 2] [--out FILE]

Median and fastest of individually synchronised calls (the GPU may be shared, and one delayed call would dominate a
mean), for each of: transcribe and transcribe_with_timestamps from device PCM and from pinned host PCM; mel + forward
+ ctc_greedy_decode_with_timestamps composed (the reference CLI's route to word timestamps); mel + forward +
ctc_greedy_decode_with_confidence composed (the CTC head writing logits, then argmax and the row statistics: the
route the fused call would take without the softmax-sum epilogue).  The calls are timed in `rounds` passes over the
list, so drift of a shared GPU shows as a spread between passes.  Then, in a separate profiled run (torch.profiler,
CUDA activities), the device time per call of the CTC-head launch with the argmax epilogue (transcribe) and with the
softmax-sum epilogue (transcribe_with_timestamps), and of the decode kernels that follow each.  Seed 1234 PCM,
random-init weights (seed 0), sequential scan.  The card's name and power limit are read in the same run and stored
with the results.  --out FILE also writes the JSON to FILE.
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "velocity-asr_b200"))
sys.path.insert(0, os.path.join(HERE, "..", "tests"))
import velocity_asr as va  # noqa: E402
import fixtures_util as FU  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=15)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--seconds", type=float, default=15.0)
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


def timed(fn, n):
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return ts


assert torch.cuda.is_available(), "timestamps_bench needs a CUDA device"
torch.manual_seed(0)
model = va.VELOCITYASR(va.VelocityASRConfig(scan_mode="sequential")).cuda().eval()
pcm = FU.synth_audio(a.batch, int(16000 * a.seconds), seed=1234).cuda()
pcm_host = pcm.cpu().pin_memory()
name, power = card()
out = {"what": f"median and fastest of {a.reps} x {a.rounds} individually synchronised calls, ms",
       "gpu": name, "power_limit": power,
       "pcm": f"{a.batch} x {a.seconds:g} s PCM (seed 1234), random-init weights (seed 0), scan_mode=sequential"}

calls = {
    "transcribe_device": lambda: model.transcribe(pcm),
    "transcribe_host": lambda: model.transcribe(pcm_host),
    "transcribe_with_timestamps_device": lambda: model.transcribe_with_timestamps(pcm),
    "transcribe_with_timestamps_host": lambda: model.transcribe_with_timestamps(pcm_host),
    "mel_forward_greedy_timestamps": lambda: va.ctc_greedy_decode_with_timestamps(
        model(va.compute_mel_spectrogram(pcm))),
    "mel_forward_greedy_confidence": lambda: va.ctc_greedy_decode_with_confidence(
        model(va.compute_mel_spectrogram(pcm))),
}
res_ts = model.transcribe_with_timestamps(pcm)
res_tr = model.transcribe(pcm)
res_cf = calls["mel_forward_greedy_confidence"]()
res_gt = calls["mel_forward_greedy_timestamps"]()
out["tokens_equal_transcribe"] = [r.tokens for r in res_ts] == res_tr
out["timestamps_equal_composed"] = [(r.tokens, r.timestamps) for r in res_ts] == [(t, s) for t, s in res_gt]
out["host_equals_device"] = model.transcribe_with_timestamps(pcm_host) == res_ts
out["tokens_total"] = sum(len(r.tokens) for r in res_ts)
d = [abs(x.log_prob - y.log_prob) / max(abs(y.log_prob), 1.0) for x, y in zip(res_ts, res_cf)]
out["log_prob_rel_diff_fused_vs_logits_route_max"] = max(d)
for fn in calls.values():         # warm-up: module loads, workspace sizes, pinned buffers
    fn()
torch.cuda.synchronize()
ts = {k: [] for k in calls}
for r in range(a.rounds):
    for k, fn in calls.items():
        t = timed(fn, a.reps)
        ts[k] += t
        out[f"{k}_round{r}_median_ms"] = round(statistics.median(t) * 1e3, 3)
for k, t in ts.items():
    out[f"{k}_ms"] = round(statistics.median(t) * 1e3, 3)
    out[f"{k}_fastest_ms"] = round(min(t) * 1e3, 3)

# device time of the kernels of interest, per call, from a profiled run of its own
from torch.profiler import ProfilerActivity, profile  # noqa: E402
PATTERNS = {
    "head_amax": r"gemm_tc2_kernel<0, false, false, false, (true|false), 128, 3>",
    "head_amax_asum": r"gemm_tc2_kernel<0, false, false, false, (true|false), 128, 11>",
    "ctc_collapse": r"ctc_collapse_kernel<true>",
    "ctc_confidence_parts": r"ctc_confidence_kernel<true>",
    "ctc_confidence_stats": r"ctc_confidence_kernel<false>",
    "argmax": r"argmax_kernel",
    "beam_rows": r"beam_rows_kernel",
}
N_PROF = 5
for k in ("transcribe_device", "transcribe_with_timestamps_device", "mel_forward_greedy_confidence"):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(N_PROF):
            calls[k]()
        torch.cuda.synchronize()
    sums = {}
    for e in prof.key_averages():
        for tag, pat in PATTERNS.items():
            if re.search(pat, e.key):
                sums[tag] = sums.get(tag, 0.0) + e.device_time_total
    for tag, us in sorted(sums.items()):
        out[f"profile_{k}_{tag}_us_per_call"] = round(us / N_PROF, 1)
print(json.dumps(out))
if a.out:
    with open(a.out, "w") as f:
        f.write(json.dumps(out, indent=1) + "\n")
