#!/usr/bin/env python
"""bench.py — RTFx of the VELOCITY-ASR v2 inference path (PCM -> log-mel -> model -> greedy CTC).

    python bench.py --gpus 1 --steps 10 --warmup 3                 # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1 # the reference's CPU path

Workload (BASELINE.json configs[1]): 64 x 15 s synthetic 16 kHz utterances per GPU, FP32,
random-init weights (torch.manual_seed(0)), audio randn*0.1 (seed 1234).  Weak scaling: every
rank processes its own 64 utterances (N = 8 is configs[2], 512 utterances); no collective on the
data path.  A "step" is one pass of the whole path over the rank's batch.

  value  = audio-seconds per wall-second with PCM already resident in HBM (vasr_transcribe),
           timed with CUDA events, max over ranks.
  e2e    = same metric through the public API with HOST buffers (VELOCITYASR.transcribe_batches over
           pinned tensors): host->device copy of the PCM and device->host copy of the token ids
           inside the timed region, every step, overlapped with the previous / next step's kernels;
           e2e.single_call is one blocking VELOCITYASR.transcribe(host tensor) per step.
  roofline = the selective-scan kernel (the kernel BASELINE.json's metric names): algorithmic
           bytes per launch (SURVEY.md section 8d: 4*(4*Di + 2*N) = 6,656 B per token-layer with
           the silu(z) gate fused) / average launch duration from CUDA events on the launch stream;
           frac = against the measured HBM copy peak, fp32_issue_frac = against the kernel's real bound
           (1,152 packed fp32 warp-instructions x 2 clocks per token-layer over 148 x 4 sub-partitions
           at the SM clock sampled during the run); traffic = DRAM bytes of one launch from the tracked
           ncu capture profiles/scan_ncu.json (tools/measure_pass.sh regenerates it).
  cpu_baseline = the reference's own PyTorch CPU path (baseline/_ref, kind "reference"; falls
           back to the numpy oracle port) on a bounded sample, rank 0 at N = 1 only; .config1 =
           BASELINE config 1 (1 x 10 s) in both scan modes.
  parity  = outside the timed region: the token ids the GPU path produced for the first utterances of
           input set 0 against the ones the cpu_baseline leg decodes for the same utterances.
  config.default_scan_mode_ms_per_step = the same step with scan_mode="parallel" (the reference's
           default semantics, configs/model.yaml:64); the headline uses "sequential" (true recurrence,
           the reference's fastest CPU mode; its parallel mode cannot run 64 utterances on this host).
  --global-batch G : strong scaling (BASELINE configs[2]): G utterances split over the ranks.
  --quantized      : BASELINE configs[4] semantics (quantize.py FakeQuantize model), same timing.
  --dump-outputs D : after the timed steps, what the last one returned (see dump_outputs) as D/<name>.npy, so that
           two builds can be compared output for output; the inputs are seeded, so equal arguments mean equal inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True     # the tree may be read-only: the benchmark writes nothing into it

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "velocity-asr_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

SR = 16000
UTT_SECONDS = 15
BATCH_PER_GPU = 64
SCAN_MODE = "sequential"      # true recurrence; see DESIGN.md (the reference's 'parallel' needs ~1 GB/utt on CPU)
METRIC = "rtfx"
UNIT = "audio-seconds/second"
WORKLOAD = "configs[1]: batch 64 x 15 s synthetic 16 kHz utterances per GPU, FP32, mel->SSM->attention->CTC greedy"


def synth_audio(batch, samples, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, samples, generator=g) * 0.1


# ----------------------------------------------------------------------------- clocks -----
class ClockSampler:
    """nvidia-smi sampled every 20 ms (B200_PROFILING.md); only samples that arrive between mark_begin()
    and mark_end() — the timed region — are reported, so idle clocks before / after it do not count."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            time.sleep(0.15)               # let the first samples arrive before the region starts
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def collect(rows):
            sm, mx, reasons = [], [], set()
            for _, r in rows:
                try:
                    sm.append(float(r[0]))
                    mx.append(float(r[1]))
                    for n, v in zip(names, r[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(n)
                except Exception:
                    pass
            return sorted(sm), mx, reasons
        inside = [x for x in self.rows if self.t0 is not None and self.t0 <= x[0] <= (self.t1 or 1e30) + 0.02]
        sm, mx, reasons = collect(inside)
        where = "timed region"
        if not sm:                          # region shorter than the sampling period: nearest samples
            sm, mx, reasons = collect(self.rows)
            where = "whole run (timed region shorter than the sampling period)"
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": where}


# The contract is ONE JSON line on stdout.  Libraries print there too (NCCL announces its version on the first
# communicator), so file descriptor 1 points at stderr while the benchmark runs and is restored for the line.
_REAL_STDOUT = None


def quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, tokens, lens):
    """What a caller of the timed path receives for its batch: tokens.npy (B, L) the greedy-CTC ids, -1 past each
    utterance's count, and lengths.npy (B,) the counts, both float32 (ids and counts are exact in it).  Should that
    exceed 64 MB, a fixed seeded sample of utterances; rows.npy names the rows written."""
    import numpy as np
    tokens, lens = np.asarray(tokens), np.asarray(lens)
    tokens = np.where(np.arange(tokens.shape[1]) < lens[:, None], tokens, -1)
    rows = np.arange(len(lens))
    per_row = 4 * (tokens.shape[1] + 2)
    if per_row * len(rows) > DUMP_LIMIT_BYTES - 4096:            # 4 KB: the three .npy headers
        keep = (DUMP_LIMIT_BYTES - 4096) // per_row
        rows = np.sort(np.random.RandomState(0).choice(len(rows), keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("tokens", tokens[rows]), ("lengths", lens[rows]), ("rows", rows)):
        np.save(os.path.join(out_dir, name + ".npy"), arr.astype(np.float32))


# ----------------------------------------------------------------------------- reference ---
def load_reference_impl():
    """(kind, module): the unmodified reference if it travelled with the repo, else None."""
    try:
        from refload import load_reference
        ref = load_reference()
        if ref is not None:
            return "reference", ref
    except Exception:
        pass
    return "port", None


def cpu_path_rtfx(n_utt, seconds, repeats, scan_mode, keep_tokens=False, batch_of=0):
    """Reference CPU path (compute_mel_spectrogram -> model -> ctc_greedy_decode, eval, no_grad,
    all host threads) on n_utt utterances; falls back to the numpy oracle port."""
    import numpy as np
    import torch
    kind, ref = load_reference_impl()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # the first n_utt utterances of the batch the GPU arm times as input set 0 (same generator stream)
    audio = synth_audio(max(n_utt, batch_of), SR * seconds, 1234)[:n_utt].contiguous()
    best = None
    if ref is not None:
        torch.manual_seed(0)
        model = ref.VELOCITYASR(ref.VelocityASRConfig(scan_mode=scan_mode)).eval()

        def run(detail=None):
            with torch.no_grad():
                mel = ref.compute_mel_spectrogram(audio)
                logits = model(mel)
                if detail is not None:          # parity material (untimed call): per-frame choice and its margin
                    top2 = logits.topk(2, dim=-1).values
                    detail["argmax"] = logits.argmax(-1).numpy()
                    detail["margin"] = (top2[..., 0] - top2[..., 1]).numpy()
                return ref.ctc_greedy_decode(logits)
    else:
        import velocity_asr as va
        import velocity_oracle as O
        torch.manual_seed(0)
        sd = {k: v.numpy() for k, v in va.VELOCITYASR(va.VelocityASRConfig()).state_dict().items()}
        a = audio.numpy()

        def run(detail=None):
            if detail is None:
                return O.transcribe(a, sd, dict(scan_mode=scan_mode), dtype=np.float32)
            logits = O.forward(O.log_mel(a), sd, dict(scan_mode=scan_mode))
            top2 = np.sort(logits, axis=-1)[..., -2:]
            detail["argmax"], detail["margin"] = logits.argmax(-1), top2[..., 1] - top2[..., 0]
            return O.ctc_greedy_decode(logits)
    detail = {} if keep_tokens else None
    tokens = run(detail)                    # warm-up (lazy init, thread pools); keeps the parity material
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    best = min(times)
    out = {"value": n_utt * seconds / best, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
           "sample": f"{n_utt} x {seconds} s utterances, scan_mode={scan_mode}, best of {repeats} after 1 warm-up, "
                     f"{best:.2f} s per pass", "seconds_per_pass": best, "times": times}
    if keep_tokens:
        out["_tokens"] = [list(map(int, t)) for t in tokens]
        out["_detail"] = detail
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_utt = args.ref_utts
    kind, ref = load_reference_impl()
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    audio = synth_audio(n_utt, SR * UTT_SECONDS, 1234)
    if ref is not None:
        torch.manual_seed(0)
        model = ref.VELOCITYASR(ref.VelocityASRConfig(scan_mode=SCAN_MODE)).eval()

        def step():
            with torch.no_grad():
                return ref.ctc_greedy_decode(model(ref.compute_mel_spectrogram(audio)))
    else:
        import numpy as np
        import velocity_asr as va
        import velocity_oracle as O
        torch.manual_seed(0)
        sd = {k: v.numpy() for k, v in va.VELOCITYASR(va.VelocityASRConfig()).state_dict().items()}
        a = audio.numpy()

        def step():
            return O.transcribe(a, sd, dict(scan_mode=SCAN_MODE), dtype=np.float32)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    total = time.perf_counter() - t0
    if args.dump_outputs:
        import numpy as np
        tok = np.full((n_utt, (1 + SR * UTT_SECONDS // 160 + 1) // 2), -1, np.int32)
        for b, t in enumerate(out):
            tok[b, :len(t)] = t
        dump_outputs(args.dump_outputs, tok, [len(t) for t in out])
    value = args.steps * n_utt * UTT_SECONDS / total
    sample = (f"each step = {n_utt} of the workload's {BATCH_PER_GPU} utterances (x {UTT_SECONDS} s), "
              f"scan_mode={SCAN_MODE}, {'torch CPU (unmodified reference)' if ref is not None else 'numpy oracle port'}, "
              f"{torch.get_num_threads()} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": n_utt, "global_batch": n_utt,
                   "seconds_per_utterance": UTT_SECONDS, "tokens_per_utterance": (1 + SR * UTT_SECONDS // 160 + 1) // 2,
                   "scan_mode": SCAN_MODE, "device": "cpu"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------- own arm ----
def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


SCAN_NCU = os.path.join(ROOT, "profiles", "scan_ncu.json")


def scan_traffic(shape, default_shape):
    """DRAM bytes (read + write) of ONE launch of the local-layer scan kernel, from the tracked ncu --set full
    capture profiles/scan_ncu.json (written by tools/ncu_scan_json.py in tools/measure_pass.sh).  The capture is
    for the default workload; it must exist and match that shape, otherwise the bench stops rather than print a
    stale number.  Another --batch has no capture: traffic is null."""
    with open(SCAN_NCU) as fh:
        cap = json.load(fh)
    if list(cap["shape"]) != list(default_shape):
        raise SystemExit(f"bench.py: {SCAN_NCU} was captured for shape {cap['shape']}, the workload is {default_shape}: "
                         "re-run tools/measure_pass.sh")
    if list(shape) != list(default_shape):
        return None, cap
    return int(cap["dram_bytes_read"]) + int(cap["dram_bytes_write"]), cap


def bind_rank_to_cores(local_rank, local_world):
    """N ranks on one host: give each rank its own slice of the cores the GPU is attached to, so that the copy
    threads and the list building of 8 ranks do not migrate over (and queue on) the same cores."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cores = [64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1]
    except Exception:
        cores = sorted(os.sched_getaffinity(0))
    cores = [c for c in cores if c in os.sched_getaffinity(0)] or sorted(os.sched_getaffinity(0))
    per = max(1, len(cores) // max(1, local_world))
    mine = cores[(local_rank * per) % len(cores):][:per] or cores
    try:
        os.sched_setaffinity(0, mine)
    except Exception:
        return None
    return mine


def collapse(frame_ids, blank=0):
    """decode.py:46-69 on one utterance's per-frame choices (checker side of bench.py's parity block)."""
    out, prev = [], None
    for t in map(int, frame_ids):
        if t != blank and t != prev:
            out.append(t)
        prev = t
    return out


def run_own_arm(args):
    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist
    import velocity_asr as va
    from velocity_asr import _native
    from velocity_asr.sharding import gather_token_arrays, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback")
    cores = bind_rank_to_cores(local_rank, local_world) if (world > 1 and args.bind_cores) else None
    if world > 1:
        torch.set_num_threads(2)           # N ranks share the host: the own arm needs no intra-op CPU parallelism
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")      # the one exchange of the design: host-side transcript gather

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    strong = args.global_batch > 0
    if strong:
        lo, hi = shard_range(args.global_batch, rank, world)
        B = hi - lo
        if args.global_batch % world:
            raise SystemExit("bench.py: --global-batch must be a multiple of the number of ranks")
    else:
        B = args.batch
    S = SR * UTT_SECONDS
    torch.manual_seed(0)
    model = va.VELOCITYASR(va.VelocityASRConfig(scan_mode=SCAN_MODE))
    if args.quantized:
        model = va.prepare_model_for_qat(model)
    model = model.to(dev).eval()
    # four distinct input sets (4 x 61 MB > the 126 MB L2) rotated across steps; each step also
    # streams > 1 GB of activations, so nothing survives in L2 from one step to the next.
    n_sets = 4
    host = [synth_audio(B, S, 1234 + rank * 16 + i).pin_memory() for i in range(n_sets)]
    devb = [h.to(dev) for h in host]
    if args.quantized:          # SURVEY 5.8 recipe: calibrate the activation quantisers on one batch of the workload
        va.calibrate_model(model, [va.compute_mel_spectrogram(devb[0][:8])], device=str(dev))
    eng = model._engine(dev)
    lib = eng.lib
    T = 1 + S // 160
    L = (T + 1) // 2
    tokens = torch.empty(B, L, dtype=torch.int32, device=dev)
    lens = torch.empty(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(stream.cuda_stream)

    def step_dev(i, handle=None):
        _native.check(lib.vasr_transcribe(handle or eng.handle, _native.ptr(devb[i % n_sets]), B, S,
                                          _native.ptr(tokens), _native.ptr(lens), sp))

    def timed_steps(handle=None):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            step_dev(i, handle)
        e1.record(stream)
        return e0, e1

    # ---- device-resident throughput
    for i in range(args.warmup):
        step_dev(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.vasr_kernel_launches(eng.handle)
    sampler.mark_begin()
    e0, e1 = timed_steps()
    barrier()
    sampler.mark_end()
    dev_ms = e0.elapsed_time(e1)
    launches = lib.vasr_kernel_launches(eng.handle) - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tokens.cpu().numpy(), lens.cpu().numpy())

    # ---- parity material: what the timed path produces for the first utterances of input set 0
    step_dev(0)
    torch.cuda.synchronize()
    n_par = min(args.cpu_utts, B)
    tok_h, len_h = tokens[:n_par].cpu().numpy(), lens[:n_par].cpu().tolist()
    gpu_tokens = [tok_h[b, :n].tolist() for b, n in enumerate(len_h)]
    gpu_argmax = model(va.compute_mel_spectrogram(devb[0][:n_par])).argmax(-1).cpu().numpy()

    # ---- scan kernel timing (separate pass so event pairs do not perturb the number above)
    lib.vasr_set_timing(eng.handle, 1)
    scan_ms, n_scan = [], 0
    for i in range(max(3, min(args.steps, 10))):
        step_dev(i)
        torch.cuda.synchronize()
        sm, sl, tot = ctypes.c_float(), ctypes.c_int32(), ctypes.c_float()
        _native.check(lib.vasr_last_timing(eng.handle, ctypes.byref(sm), ctypes.byref(sl), ctypes.byref(tot)))
        scan_ms.append((sm.value, tot.value))
        n_scan = sl.value
    lib.vasr_set_timing(eng.handle, 0)

    # ---- end to end through the public API, host buffers in, token lists out.
    # (a) the streaming call: VELOCITYASR.transcribe_batches(iterable of pinned host batches) copies batch i+1
    #     host->device and batch i-1's token ids device->host while batch i computes; every step's H2D and D2H
    #     are inside the timed region.  With N > 1 every step's token ids are also gathered on the host to rank 0
    #     (velocity_asr.sharding.gather_token_arrays: fixed-size int32 arrays over a gloo group, no pickling) inside
    #     the timed region: the design's only exchange; every rank still builds the token lists of its own shard.
    #     (b) one blocking transcribe(host batch) call per step.
    if world == 1:
        for _ in model.transcribe_batches(host[i % n_sets] for i in range(max(2, args.warmup))):
            pass
    else:
        # warm-up includes the gather: the first collective on a gloo group sets up its TCP pairs (milliseconds,
        # growing with the number of ranks), which is connection set-up, not a step
        for tok_np, len_np in model.transcribe_batches((host[i % n_sets] for i in range(max(2, args.warmup))),
                                                       as_arrays=True):
            gather_token_arrays(tok_np, len_np, group=host_group, dst=0)
    barrier()
    t0 = time.perf_counter()
    n_out = n_all = 0
    if world == 1:
        for out in model.transcribe_batches(host[i % n_sets] for i in range(args.steps)):
            n_out += len(out)
        n_all = n_out
    else:
        from velocity_asr.model import _token_lists
        for tok_np, len_np in model.transcribe_batches((host[i % n_sets] for i in range(args.steps)), as_arrays=True):
            got = gather_token_arrays(tok_np, len_np, group=host_group, dst=0)
            n_out += len(_token_lists(torch.from_numpy(tok_np), torch.from_numpy(len_np)))
            n_all += got[1].shape[0] if got is not None else B * world
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert n_out == args.steps * B and n_all == args.steps * B * world
    barrier()
    for i in range(max(1, args.warmup)):
        model.transcribe(host[i % n_sets])
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        out = model.transcribe(host[i % n_sets])
    torch.cuda.synchronize()
    e2e1_s = time.perf_counter() - t0
    barrier()

    # ---- the same step under the reference's DEFAULT scan semantics (scan_mode="parallel")
    par_ms = float("nan")
    if not args.no_extras:
        torch.manual_seed(0)
        model_p = va.VELOCITYASR(va.VelocityASRConfig(scan_mode="parallel"))
        if args.quantized:
            model_p = va.prepare_model_for_qat(model_p)
            model_p._act_qparams = dict(model._act_qparams)
        model_p = model_p.to(dev).eval()
        eng_p = model_p._engine(dev)
        for i in range(args.warmup):
            step_dev(i, eng_p.handle)
        barrier()
        p0, p1 = timed_steps(eng_p.handle)
        barrier()
        par_ms = p0.elapsed_time(p1)

    times = torch.tensor([dev_ms, e2e_s * 1e3, e2e1_s * 1e3, par_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, e2e1_ms, par_ms = (float(t) for t in times)

    if rank == 0:
        audio_s = world * B * UTT_SECONDS * args.steps
        cfg = model.config
        di = cfg.d_model * cfg.ssm_expand_ratio
        # local scan launches come first in each step; the 2 global launches (93 tokens) are tiny
        local_bytes = B * L * 4 * (4 * di + 2 * cfg.ssm_state_dim)
        K1 = min(max(64, L // 8), L)
        global_bytes = B * K1 * 4 * (4 * 2 * cfg.d_model + 2 * cfg.global_ssm_state_dim)
        scan_total_ms = sum(s for s, _ in scan_ms) / len(scan_ms)
        step_total_ms = sum(t for _, t in scan_ms) / len(scan_ms)
        all_bytes = cfg.ssm_layers * local_bytes + cfg.global_ssm_layers * global_bytes
        # per-launch average over the local-layer launches: apportion the measured total by bytes
        local_ms = scan_total_ms * (cfg.ssm_layers * local_bytes / all_bytes) / cfg.ssm_layers
        peak, peak_src = hbm_peak()
        achieved = local_bytes / (local_ms * 1e-3) / 1e9
        traffic, cap = scan_traffic((B, L, di, cfg.ssm_state_dim), (BATCH_PER_GPU, L, di, cfg.ssm_state_dim))
        # fp32-issue bound: 3 fp32 operations per (state, step) = Di*N*3/2/32 packed warp-instructions per token-layer,
        # each holding a sub-partition's FMA pipe for 2 clocks; 148 SMs x 4 sub-partitions at the sampled SM clock
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        packed_instr = di * cfg.ssm_state_dim * 3 // 2 // 32
        issue_floor_ms = B * L * packed_instr * 2 / (148 * 4 * sm_mhz * 1e6) * 1e3
        line = {
            "metric": METRIC, "value": audio_s / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD if not args.quantized else WORKLOAD + " [quantize.py FakeQuantize model, "
                       "BASELINE configs[4] semantics]",
                       "batch_per_gpu": B, "global_batch": B * world,
                       "seconds_per_utterance": UTT_SECONDS, "tokens_per_utterance": L, "scan_mode": SCAN_MODE,
                       "default_scan_mode_ms_per_step": None if par_ms != par_ms else par_ms / args.steps,
                       "default_scan_mode": "parallel (configs/model.yaml:64, ssm.py:216-295): same weights and input, "
                                            "scan_quirk kernel in the 8 local layers",
                       "parallelism": f"dp{world} (utterance shards, no data-path collective)",
                       "l2": "4 rotating input sets (244 MB) + >1 GB of activations per step: larger than L2"},
            "e2e": {"value": audio_s / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": B * S * 4, "d2h_bytes_per_step": B * L * 4 + B * 4,
                    "api": "VELOCITYASR.transcribe_batches(pinned host batches) -> List[List[int]] per batch "
                           "(H2D of batch i+1 and D2H of batch i-1 overlap the kernels of batch i)"
                           + ("; + sharding.gather_token_arrays of every step's token ids to rank 0 (gloo, host)"
                              if world > 1 else ""),
                    "single_call": {"value": audio_s / (e2e1_ms * 1e-3), "ms_per_step": e2e1_ms / args.steps,
                                    "api": "VELOCITYASR.transcribe(pinned host tensor), one blocking call per step"}},
            "gpu_launches": int(launches),
            "roofline": {"kernel": cap.get("kernel", "scan_seq_kernel") + " (8 local SSM layers)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src,
                         "fp32_issue_frac": issue_floor_ms / local_ms, "fp32_issue_floor_ms": issue_floor_ms,
                         "fp32_issue_model": f"{packed_instr} packed fp32 warp-instructions x 2 clocks per token-layer / "
                                             f"(148 SMs x 4 sub-partitions x {sm_mhz:.0f} MHz)",
                         "traffic": traffic, "traffic_source": os.path.relpath(SCAN_NCU, ROOT) + ": " + cap.get("source", ""),
                         "algorithmic_bytes_per_launch": local_bytes, "avg_launch_ms": local_ms,
                         "scan_launches_per_step": n_scan, "scan_ms_per_step": scan_total_ms,
                         "scan_share_of_step": scan_total_ms / step_total_ms,
                         "note": "the kernel is fp32-issue / shared-memory-delivery bound, not HBM bound (DESIGN.md): "
                                 "frac is the honest HBM fraction of algorithmic bytes, fp32_issue_frac the fraction of "
                                 "its real ceiling"},
            "clocks": clocks,
        }
        if world > 1 and cores:
            line["config"]["cores_per_rank"] = len(cores)
        if world == 1 and not args.no_cpu_baseline:
            try:
                base = cpu_path_rtfx(n_par, UTT_SECONDS, 2, SCAN_MODE, keep_tokens=True, batch_of=B)
                ref_tokens, det = base.pop("_tokens"), base.pop("_detail")
                line["cpu_baseline"] = base
                equal = sum(int(a == b) for a, b in zip(gpu_tokens, ref_tokens))
                # frames the reference itself cannot call: best-minus-second margin of ITS logits <= 1e-4 (its own
                # fp32 rounding noise is ~1e-5 at |logit| ~ 2).  Everywhere else the per-frame choice must agree, and
                # with those frames pinned to the reference's choice the collapsed token lists must be identical.
                near = det["margin"] <= 1e-4
                same = gpu_argmax == det["argmax"]
                pinned = np.where(near, det["argmax"], gpu_argmax)
                equal_pinned = sum(int(collapse(p) == r) for p, r in zip(pinned, ref_tokens))
                line["parity"] = {"utts": len(ref_tokens), "tokens_equal": equal,
                                  "tokens_equal_near_ties_pinned": equal_pinned,
                                  "frames": int(same.size), "frames_equal": int(same.sum()),
                                  "near_tie_frames": int(near.sum()),
                                  "frames_differing_off_near_ties": int((~same & ~near).sum()),
                                  "what": "greedy-CTC token lists of the first utterances of input set 0: the timed GPU "
                                          f"path vs the cpu_baseline leg ({base['kind']}), outside the timed region; a "
                                          "near-tie frame has a best-minus-second margin <= 1e-4 in the reference's own "
                                          "fp32 logits (random-init logits are nearly flat)"}
                if args.quantized:
                    line["parity"]["note"] = "cpu leg runs the FP32 reference model; the GPU arm is the FakeQuantize model"
                if not args.no_extras:
                    c1 = {}
                    for mode in ("sequential", "parallel"):
                        r = cpu_path_rtfx(1, 10, 3, mode)
                        c1[mode] = {"value": r["value"], "seconds_per_pass": r["seconds_per_pass"]}
                    line["cpu_baseline"]["config1"] = dict(
                        c1, what="BASELINE configs[0]: 1 x 10 s, mel + forward + greedy on the host cores, best of 3")
            except Exception as exc:  # the baseline must never sink the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                                        "sample": f"failed: {exc!r}"}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="utterances per GPU")
    ap.add_argument("--cpu-utts", type=int, default=16, help="utterances in the cpu_baseline sample")
    ap.add_argument("--ref-utts", type=int, default=BATCH_PER_GPU,
                    help="utterances per step of --impl reference (default: the workload's 64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the default-scan-mode timing and the config-1 CPU figures")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: this many utterances in total, split over the ranks (configs[2]: 512)")
    ap.add_argument("--quantized", action="store_true", help="time the FakeQuantize model (configs[4] semantics)")
    ap.add_argument("--bind-cores", action="store_true", help="N > 1: pin each rank to its share of the GPU's cores")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0's shard when N > 1)")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    quiet_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_own_arm(args)


if __name__ == "__main__":
    main()
