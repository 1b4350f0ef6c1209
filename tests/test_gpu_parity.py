"""Parity of the CUDA path (through the C ABI of libvasr.so) with the reference.

Checked against (1) golden fixtures produced by running the reference (tests/golden), (2) the
numpy oracle on fresh seeded inputs, (3) size-independent properties at BASELINE sizes.
Tolerances (BASELINE.json north_star): mel 1e-4 absolute; activations / logits 1e-3 relative
to the tensor's max magnitude (fp32 path: observed ~1e-5); token ids bit-exact.
"""
import os

import numpy as np
import pytest
import torch

import fixtures_util as FU
import velocity_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LOGIT_RTOL = 1e-3
MEL_ATOL = 1e-4


@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


def rel(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a.astype(np.float64) - b).max() / (np.abs(b).max() + 1e-30))


def make_model(va, mode, amp=False):
    torch.manual_seed(FU.WEIGHT_SEED)
    m = va.VELOCITYASR(va.VelocityASRConfig(scan_mode=mode))
    if amp:
        m.load_state_dict(FU.amplify_state_dict(m.state_dict()))
    return m.cuda().eval()


def np_sd(m):
    return {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}


# ------------------------------------------------------------------ projections ----------
@pytest.mark.parametrize("M,K,N,act", [(1, 16, 1, None), (130, 192, 768, None), (257, 384, 512, "softplus"),
                                       (100, 192, 1000, None), (300, 48, 192, None), (64, 240, 192, "gelu"),
                                       (513, 400, 402, None), (77, 384, 48, "sigmoid")])
def test_linear(va, M, K, N, act):
    g = torch.Generator().manual_seed(M * 7 + N)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    y = va.linear(x.cuda(), w.cuda(), b.cuda(), activation=act)
    ref = O.linear(x.double().numpy(), w.double().numpy(), b.double().numpy())
    ref = {None: lambda v: v, "gelu": O.gelu, "softplus": O.softplus, "sigmoid": O.sigmoid}[act](ref)
    assert y.shape == (M, N)
    assert rel(y, ref) < 2e-6
    y2 = va.linear(x.cuda(), w.cuda())          # no bias
    assert rel(y2, O.linear(x.double().numpy(), w.double().numpy())) < 2e-6


@pytest.mark.parametrize("M,K,N,act", [(128, 32, 128, None), (1000, 192, 768, None), (5000, 384, 512, "softplus"),
                                       (700, 48, 192, None), (513, 240, 192, "gelu"), (130, 192, 1000, None),
                                       (3000, 384, 192, "sigmoid"), (48064, 192, 384, "gelu")])
def test_linear_tensor_cores(va, M, K, N, act):
    """tcgen05 / TMEM / TMA projection kernel with the 3xTF32 split: fp32-grade accuracy."""
    g = torch.Generator().manual_seed(M + 3 * N)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    y = va.linear(x.cuda(), w.cuda(), b.cuda(), activation=act, tensor_cores=True)
    ref = O.linear(x.double().numpy(), w.double().numpy(), b.double().numpy())
    ref = {None: lambda v: v, "gelu": O.gelu, "softplus": O.softplus, "sigmoid": O.sigmoid}[act](ref)
    assert y.shape == (M, N)
    assert rel(y, ref) < 5e-6
    y_simt = va.linear(x.cuda(), w.cuda(), b.cuda(), activation=act) if K % 16 == 0 else None
    if y_simt is not None:
        assert rel(y, y_simt.double().cpu().numpy()) < 5e-6


def test_model_runs_on_tensor_cores(va, golden):
    """The token-sized projections of a forward pass go through the tcgen05 kernel."""
    from velocity_asr import _native
    m = make_model(va, "sequential")
    mel = torch.randn(4, 401, 80, device="cuda")
    m(mel)
    eng = m._engine(mel.device)
    assert _native.lib().vasr_tc_launches(eng.handle) >= 8 * 5


# ------------------------------------------------------------------ front end ------------
def test_log_mel_golden(va, golden):
    g = golden("frontend")
    audio = FU.synth_audio(2, 16000).cuda()
    mel = va.compute_mel_spectrogram(audio)
    assert mel.shape == (2, 101, 80)
    assert np.abs(mel.cpu().numpy() - g["mel"]).max() < MEL_ATOL
    raw = va.compute_mel_spectrogram(audio, normalize=False)
    assert np.abs(raw.cpu().numpy() - g["mel_raw"]).max() < MEL_ATOL
    odd = va.compute_mel_spectrogram(FU.synth_audio(3, 4037, seed=99).cuda())
    assert odd.shape == (3, 26, 80)
    assert np.abs(odd.cpu().numpy() - g["mel_odd"]).max() < MEL_ATOL
    one = va.compute_mel_spectrogram(audio[0, :800])
    assert one.shape == (6, 80)
    assert np.abs(one.cpu().numpy() - g["mel_1d"]).max() < MEL_ATOL


def test_log_mel_oracle_15s(va, golden):
    g = golden("frontend")
    audio = FU.synth_audio(3, 240000, seed=5)
    mel = va.compute_mel_spectrogram(audio.cuda())
    assert mel.shape == (3, 1501, 80)
    ref = O.log_mel(audio.numpy(), filters=g["filterbank"], window=g["window"])
    assert np.abs(mel.cpu().numpy() - ref).max() < MEL_ATOL
    # per (utterance, bin): zero mean, unit unbiased std over time (audio.py:132-135)
    assert mel.mean(1).abs().max() < 1e-4
    assert (mel.std(1) - 1).abs().max() < 1e-4


def test_log_mel_rejects_short_and_stages_host_input(va):
    with pytest.raises(RuntimeError):
        va.compute_mel_spectrogram(torch.zeros(1, 150).cuda())     # reflect pad needs > 200 samples
    audio = FU.synth_audio(2, 8000, seed=5)
    host = va.compute_mel_spectrogram(audio)                        # CPU tensor: staged to the GPU, result back on CPU
    assert host.device.type == "cpu"
    assert torch.equal(host, va.compute_mel_spectrogram(audio.cuda()).cpu())   # same kernels, same bits


def test_reference_smoke_script_sequence_runs_unchanged(va):
    """/root/reference/test_vel.py:12-47 verbatim in its calls: model, input and logits never leave the CPU
    on the caller's side (the kernels still run on the GPU: host tensors are staged)."""
    from velocity_asr import VELOCITYASR, VelocityASRConfig, ctc_greedy_decode
    config = VelocityASRConfig()
    model = VELOCITYASR(config)
    assert model.count_parameters() > 0
    batch_size, num_frames, mel_bins = 2, 500, 80
    torch.manual_seed(3)
    x = torch.randn(batch_size, num_frames, mel_bins)
    model.eval()
    with torch.no_grad():
        logits = model(x)
    assert logits.device.type == "cpu" and tuple(logits.shape) == (batch_size, (num_frames + 1) // 2, config.vocab_size)
    decoded = ctc_greedy_decode(logits)
    assert len(decoded) == batch_size
    # the staged call is the CUDA call
    on_gpu = model.cuda()(x.cuda())
    assert torch.equal(on_gpu.cpu(), logits)
    assert ctc_greedy_decode(on_gpu) == decoded


def test_reference_transcribe_loop_body_runs_unchanged(va):
    """The body of transcribe_file (scripts/transcribe.py:69-126) with its own calls and argument devices: mel
    computed from a CPU waveform, moved to the model's device, greedy decode with and without timestamps, word
    assembly.  Checked against the fused transcribe() and the oracle's run decoder."""
    from velocity_asr import (VELOCITYASR, VelocityASRConfig, CTCDecoder, compute_mel_spectrogram,
                              create_default_vocabulary, ctc_greedy_decode_with_timestamps, words_with_timestamps,
                              frames_to_seconds)
    from velocity_asr.audio import SAMPLE_RATE, HOP_LENGTH
    assert (SAMPLE_RATE, HOP_LENGTH) == (16000, 160)
    device = "cuda"
    torch.manual_seed(0)
    model = VELOCITYASR(VelocityASRConfig(scan_mode="sequential"))
    model.load_state_dict(FU.amplify_state_dict(model.state_dict()))
    model = model.to(device).eval()
    decoder = CTCDecoder(create_default_vocabulary(model.config.vocab_size))
    audio = FU.synth_audio(1, 3 * 16000, seed=17)[0]                # what load_audio returns: 1-D CPU waveform
    mel = compute_mel_spectrogram(audio)
    assert mel.device.type == "cpu" and mel.dim() == 2
    with torch.no_grad():
        mel_tensor = mel.unsqueeze(0).to(device)
        logits = model(mel_tensor)
        tokens, timestamps = ctc_greedy_decode_with_timestamps(logits)[0]
        text = decoder.decode_greedy(logits)[0]
    assert tokens == model.transcribe(audio.to(device))[0]
    o_tokens, o_times = O.ctc_greedy_decode_with_timestamps(logits.cpu().numpy())[0]
    assert tokens == o_tokens and timestamps == [tuple(t) for t in o_times]
    assert text == decoder._tokens_to_text(tokens)
    words = words_with_timestamps(tokens, timestamps, decoder.vocabulary)
    assert " ".join(w["word"] for w in words).split() == "".join(
        decoder.vocabulary[t] for t in tokens).replace("▁", " ").split()
    for w in words:
        assert 0.0 <= w["start"] <= w["end"] <= frames_to_seconds(logits.size(1))


# ------------------------------------------------------------------ selective scan -------
def test_scan_golden(va, golden):
    g = golden("scan_ops")
    for case in g["cases"]:
        name, b, L, di, n, seed, st = eval(case)
        x, dt, A, Bm, Cm, D = [torch.from_numpy(a).cuda() for a in FU.scan_inputs(b, L, di, n, seed, st)]
        ys = va.selective_scan(x, dt, A, Bm, Cm, D, scan_mode="sequential")
        yp = va.selective_scan(x, dt, A, Bm, Cm, D, scan_mode="parallel")
        assert rel(ys, g[name + "_seq"]) < 1e-4, name
        assert rel(yp, g[name + "_par"]) < 1e-4, name
        ym = va.selective_scan(x, dt, A, Bm, Cm, D, scan_mode="mamba")
        assert torch.equal(ym, ys)


@pytest.mark.parametrize("n,structured,di", [
    pytest.param(n, s, di, id=f"{n}-{s}" + (f"-di{di}" if di != 128 else ""))
    for n, s, di in [(64, True, 128), (64, False, 128), (32, True, 128), (32, False, 128), (16, True, 128),
                     (16, False, 128),                  # the unstructured-A kernels of N = 16
                     (16, False, 64), (32, True, 192)]])  # 1-warp (N = 16) and 2-warp (N = 32) CTAs of the recurrence
@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_scan_oracle(va, n, structured, di, mode):
    L = 203 if mode == "sequential" else 71            # not a multiple of the 32-step chunk / of 8
    x, dt, A, Bm, Cm, D = FU.scan_inputs(2, L, di, n, 100 + n, structured)
    rs = np.random.RandomState(3)
    z = rs.standard_normal(x.shape).astype(np.float32)
    t = lambda a: torch.from_numpy(a).cuda()
    y = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode=mode)
    d = lambda a: a.astype(np.float64)
    ref = O.selective_scan(d(x), d(dt), d(A), d(Bm), d(Cm), d(D), mode) * O.silu(d(z))
    assert rel(y, ref) < 1e-4
    y0 = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), None, scan_mode=mode)   # no skip, no gate
    assert rel(y0, O.selective_scan(d(x), d(dt), d(A), d(Bm), d(Cm), None, mode)) < 1e-4
    if n == 64 and structured and mode == "sequential":
        # y rows 8-byte but not 16-byte aligned (ldy = Di + 2): the row-packed kernel declines them, and the
        # structured recurrence kernel takes them (scan_seq_kernel<4, 4, 2, true>, which no other call reaches)
        import ctypes
        from velocity_asr import _native
        B, Lx, Di = x.shape
        xs, dts, As, Bs, Cs, Ds, zs = (t(a) for a in (x, dt, A, Bm, Cm, D, z))
        ys = torch.full((B * Lx + 1, Di + 2), float("nan"), device="cuda")
        _native.check(_native.lib().vasr_selective_scan(
            _native.ptr(xs), Di, _native.ptr(dts), Di, _native.ptr(As), _native.ptr(Bs), n, _native.ptr(Cs), n,
            _native.ptr(Ds), _native.ptr(zs), Di, _native.ptr(ys), Di + 2, B, Lx, Di, n, 0,
            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
        got = ys.cpu().numpy()
        assert rel(got[:B * Lx, :Di].reshape(B, Lx, Di), ref) < 1e-4
        assert np.isnan(got[:, Di:]).all() and np.isnan(got[B * Lx:]).all()


def test_scan_scaled_state_extremes(va):
    """The structured-A kernel carries the state divided by u = x*dt (scan.cu): exact zeros, denormal-sized and
    huge inputs, sign flips and long zero runs must not disturb it."""
    rs = np.random.RandomState(12)
    B, L, Di, N = 2, 150, 384, 64
    x, dt, A, Bm, Cm, D = FU.scan_inputs(B, L, Di, N, seed=31, structured_a=True)
    x[:, 10:40, :128] = 0.0                                   # a long run of exact zeros
    x[:, 50:60, 128:256] *= 1e-25                             # |u| far below the clamp
    x[:, 70:75, 256:] *= 1e4                                  # large inputs, then back to O(1)
    x[1, :, ::7] = 0.0                                        # rows that are zero throughout
    dt[:, 90:95] = 1e-6                                       # tiny step sizes (decay ~ 1)
    z = rs.standard_normal(x.shape).astype(np.float32)
    ref = O.selective_scan(x.astype(np.float64), dt.astype(np.float64), A.astype(np.float64), Bm.astype(np.float64),
                           Cm.astype(np.float64), D.astype(np.float64), mode="sequential") * (z / (1 + np.exp(-z.astype(np.float64))))
    t = lambda a: torch.from_numpy(a).cuda()
    got = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode="sequential").cpu().numpy()
    assert np.isfinite(got).all()
    scale = np.abs(ref).max(axis=(1,), keepdims=True) + 1e-6   # per (batch, channel): rows differ by 1e4 in magnitude
    assert (np.abs(got - ref) / scale).max() < 1e-4        # the bar of test_scan_oracle, here per channel
    zero_rows = np.abs(x[1]).max(axis=0) == 0
    assert np.abs(got[1][:, zero_rows]).max() < 1e-9            # y = 0 (up to the 1e-12 clamp) where x is 0 throughout


@pytest.mark.parametrize("B,L", [(64, 130), (50, 20), (50, 16), (75, 49), (150, 33)])
def test_scan_large_batch_time_split(va, B, L):
    """The large-batch kernel (row pairs per packed register, time axis cut into slots that hand the state over
    through global memory; scan.cu, scan_rp_kernel) against the oracle: shapes where a slot holds a fraction of a
    chain (64 x 130: 5.8 chunks of 9 per slot), about one chunk (50 x 20), whole chains only (50 x 16: no
    hand-over) or several chains plus two fractions (150 x 33), with the extremes of test_scan_scaled_state_extremes
    placed across the cuts."""
    Di, N = 384, 64
    x, dt, A, Bm, Cm, D = FU.scan_inputs(B, L, Di, N, seed=500 + B + L, structured_a=True)
    x[:, 3:9, :64] = 0.0
    x[:, 14:18, 64:128] *= 1e-25                                # straddles the first chunk boundary
    x[:, min(L - 1, 30):min(L, 35), 128:192] *= 1e4
    rs = np.random.RandomState(B)
    z = rs.standard_normal(x.shape).astype(np.float32)
    t = lambda a: torch.from_numpy(a).cuda()
    got = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode="sequential")
    again = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode="sequential")
    assert torch.equal(got, again)                             # the hand-over order does not touch the arithmetic
    d = lambda a: a.astype(np.float64)
    ref = O.scan_sequential(d(x), d(dt), d(A), d(Bm), d(Cm), d(D)) * O.silu(d(z))
    got = got.cpu().numpy()
    assert np.isfinite(got).all()
    scale = np.abs(ref).max(axis=1, keepdims=True) + 1e-6
    assert (np.abs(got - ref) / scale).max() < 1e-4
    # an utterance alone (small-batch kernel, no split) gives the same numbers to fp32 rounding
    alone = va.selective_scan(t(x[:1]), t(dt[:1]), t(A), t(Bm[:1]), t(Cm[:1]), t(D), z=t(z[:1]), scan_mode="sequential")
    assert (np.abs(alone.cpu().numpy() - got[:1]) / scale[:1]).max() < 2e-5


@pytest.mark.parametrize("n,structured", [(64, True), (32, True), (64, False)])
def test_scan_parallel_mode_dead_state_shortcuts(va, n, structured):
    """The reference's 'parallel' rule multiplies every new term by exp(A cumsum(dt)); once that is an exact fp32
    zero for all rows of a CTA the kernel copies hP from the parent index (phase 2) and from the next power of two
    on emits x D only (phase 3).  Against the oracle on a sequence long enough for all three phases, with rows that
    die at different times, and bit for bit against the same rows computed next to a row that never dies (that CTA
    runs the full rule throughout)."""
    B, L, Di = 2, 700, 128
    x, dt, A, Bm, Cm, D = FU.scan_inputs(B, L, Di, n, seed=900 + n, structured_a=structured)
    dt[:, :, 32:48] *= 0.4                                     # a CTA whose rows die later than the others
    dt[1, :, 64:80] *= 0.02                                    # a CTA (batch 1, rows 64..79) that never dies
    rs = np.random.RandomState(n)
    z = rs.standard_normal(x.shape).astype(np.float32)
    t = lambda a: torch.from_numpy(a).cuda()
    got = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode="parallel")
    d = lambda a: a.astype(np.float64)
    ref = O.selective_scan(d(x), d(dt), d(A), d(Bm), d(Cm), d(D), "parallel") * O.silu(d(z))
    assert rel(got, ref) < 1e-4
    tail = got[:, 512:].cpu().numpy()                         # far beyond the decay horizon of the ordinary rows
    plain = (x * D)[:, 512:] * (z / (1 + np.exp(-z.astype(np.float64))))[:, 512:]
    assert np.abs(tail[0] - plain[0]).max() < 1e-5            # phase 3: y = x D silu(z)
    # one never-dying row per CTA of 8 or 16 rows keeps every CTA in the full rule; the other rows must not notice
    dt2 = dt.copy()
    dt2[:, :, ::8] *= 0.01
    keep = np.ones(Di, dtype=bool); keep[::8] = False
    a1 = va.selective_scan(t(x), t(dt), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode="parallel")[:, :, torch.from_numpy(keep).cuda()]
    a2 = va.selective_scan(t(x), t(dt2), t(A), t(Bm), t(Cm), t(D), z=t(z), scan_mode="parallel")[:, :, torch.from_numpy(keep).cuda()]
    assert torch.equal(a1, a2)
    with pytest.raises(ValueError):
        va.selective_scan(t(x), t(-dt), t(A), t(Bm), t(Cm), t(D), scan_mode="parallel")


def test_scan_mamba_signature(va):
    x, dt, A, Bm, Cm, D = FU.scan_inputs(2, 50, 384, 64, 77, True)
    t = lambda a: torch.from_numpy(a).cuda()
    y = va.selective_scan_fn(t(x).transpose(1, 2).contiguous(), t(dt).transpose(1, 2).contiguous(),
                             t(A).unsqueeze(0).expand(384, -1).contiguous(), t(Bm).unsqueeze(1), t(Cm).unsqueeze(1),
                             t(D))
    assert y.shape == (2, 384, 50)
    d = lambda a: a.astype(np.float64)
    assert rel(y.transpose(1, 2), O.scan_sequential(d(x), d(dt), d(A), d(Bm), d(Cm), d(D))) < 1e-4


def test_scan_properties_config2_size(va):
    """BASELINE config 2 shape (64 x 751 x 384, N = 64): causality, linearity in x, batch independence."""
    B, L, Di, N = 64, 751, 384, 64
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, L, Di, device="cuda", generator=g)
    dt = torch.nn.functional.softplus(torch.randn(B, L, Di, device="cuda", generator=g))
    Bm = torch.randn(B, L, N, device="cuda", generator=g)
    Cm = torch.randn(B, L, N, device="cuda", generator=g)
    A = -torch.arange(1, N + 1, device="cuda", dtype=torch.float32)
    D = torch.randn(Di, device="cuda", generator=g)
    y = va.selective_scan(x, dt, A, Bm, Cm, D)
    assert torch.isfinite(y).all()
    assert torch.equal(y, va.selective_scan(x, dt, A, Bm, Cm, D))                      # deterministic
    y_pre = va.selective_scan(x[:, :300].contiguous(), dt[:, :300].contiguous(), A, Bm[:, :300].contiguous(),
                              Cm[:, :300].contiguous(), D)
    assert torch.equal(y_pre, y[:, :300])                                               # causal
    y2 = va.selective_scan(2 * x, dt, A, Bm, Cm, D)
    assert (y2 - 2 * y).abs().max() <= 1e-5 * y.abs().max()                             # linear in x
    y_one = va.selective_scan(x[5:6].contiguous(), dt[5:6].contiguous(), A, Bm[5:6].contiguous(),
                              Cm[5:6].contiguous(), D)
    assert torch.equal(y_one[0], y[5])                                                  # shards independently
    sub = slice(0, 2)
    d = lambda a: a[sub].double().cpu().numpy()
    ref = O.scan_sequential(d(x), d(dt), A.double().cpu().numpy(), d(Bm), d(Cm), D.double().cpu().numpy())
    assert rel(y[sub], ref) < 1e-4


# ------------------------------------------------------------------ blocks ---------------
def test_blocks_golden(va, golden):
    g = golden("blocks")
    rs = np.random.RandomState(21)
    xin = torch.from_numpy(rs.standard_normal((2, 75, 192)).astype(np.float32)).cuda()
    xlong = torch.from_numpy(rs.standard_normal((1, 1100, 192)).astype(np.float32)).cuda()
    m = make_model(va, "sequential", amp=True)
    assert rel(m.run_ssm_block(xin, 0, "local"), g["local_block0_seq"]) < LOGIT_RTOL
    assert rel(m.run_ssm_block(xin, 0, "local", scan_mode="parallel"), g["local_block0_par"]) < LOGIT_RTOL
    assert rel(m.run_global_context(xin), g["global_context"]) < LOGIT_RTOL
    assert rel(m.run_global_context(xlong)[:, ::11], g["global_context_L1100"]) < LOGIT_RTOL
    assert rel(m.run_ctc_head(xin)[:, ::5], g["ctc_head"]) < LOGIT_RTOL
    sd = np_sd(m)
    x64 = xin.double().cpu().numpy()
    assert rel(m.run_ssm_block(xin, 3, "local"), O.ssm_block(x64, sd, "local_ssm.layers.3.", "sequential")) < 1e-4
    assert rel(m.run_ssm_block(xin, 1, "global"),
               O.ssm_block(x64, sd, "global_context.global_ssm.layers.1.", "parallel")) < 1e-4


# ------------------------------------------------------------------ whole model ----------
@pytest.mark.parametrize("mode", ["sequential", "parallel"])
@pytest.mark.parametrize("amp", [False, True])
def test_forward_golden(va, golden, mode, amp):
    g = golden("model_small")
    mel = torch.from_numpy(golden("frontend")["mel"]).cuda()
    m = make_model(va, mode, amp)
    logits, f = m(mel, return_features=True)
    tag = f"{mode}{'_amp' if amp else ''}"
    assert logits.shape == (2, 51, 1000)
    assert rel(f["temporal_binding"], g[tag + "_tb"]) < LOGIT_RTOL
    assert rel(f["local_features"], g[tag + "_local"]) < LOGIT_RTOL
    assert rel(f["fused_features"], g[tag + "_fused"]) < LOGIT_RTOL
    assert rel(logits, g[tag + "_logits"]) < LOGIT_RTOL
    toks = va.ctc_greedy_decode(logits)
    assert toks == [[int(t) for t in row if t >= 0] for row in g[tag + "_tokens"]]
    assert torch.equal(m(mel), logits)          # plain call, and run-to-run reproducible


def test_mamba_mode_equals_sequential(va, golden):
    mel = torch.from_numpy(golden("frontend")["mel"]).cuda()
    a = make_model(va, "sequential", True)(mel)
    b = make_model(va, "mamba", True)(mel)
    assert torch.equal(a, b)


def decode_with_reference_on_near_ties(va, logits, ref_argmax, safe):
    """Greedy tokens of OUR logits through OUR decoder, with the frames the reference itself cannot call
    (best-minus-second margin of the reference's own logits below the caller's threshold) pinned to its choice.  The
    result must equal the reference's token list unconditionally: every margin-safe frame is ours."""
    lg = logits.clone()
    ref = torch.from_numpy(np.asarray(ref_argmax)).to(lg.device).long()
    unsafe = torch.from_numpy(~np.asarray(safe)).to(lg.device)
    pinned = torch.full_like(lg, -1e30).scatter_(-1, ref.unsqueeze(-1), 0.0)
    lg[unsafe] = pinned[unsafe]
    return va.ctc_greedy_decode(lg)


@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_config1_end_to_end(va, golden, mode):
    """BASELINE config 1: 1 x 10 s, mel + forward + greedy."""
    g = golden("config1")
    audio = FU.synth_audio(1, 160000).cuda()
    m = make_model(va, mode)
    mel = va.compute_mel_spectrogram(audio)
    assert np.abs(mel[:, ::50].cpu().numpy() - g["mel_sub"]).max() < MEL_ATOL
    logits = m(mel)
    assert logits.shape == (1, 501, 1000)
    assert rel(logits[:, ::25], g[mode + "_logits_sub"]) < LOGIT_RTOL
    am = logits.argmax(-1).cpu().numpy()
    safe = g[mode + "_margin"] > 1e-3            # frames whose argmax is not a near-tie in the reference
    assert (am == g[mode + "_argmax"])[safe].all()
    assert (am == g[mode + "_argmax"]).mean() >= 0.99
    assert va.ctc_greedy_decode(logits)[0] == m.transcribe(audio)[0]
    assert safe.mean() > 0.99
    assert decode_with_reference_on_near_ties(va, logits, g[mode + "_argmax"], safe)[0] == g[mode + "_tokens"].tolist()
    if (am == g[mode + "_argmax"]).all():
        assert m.transcribe(audio)[0] == g[mode + "_tokens"].tolist()


@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_config2_full_batch(va, golden, mode):
    """BASELINE configs[1], the benchmarked size: the FULL 64 x 15 s seed-1234 batch bench.py times goes through
    mel + forward + greedy in one call; utterances 0, 31 and 63 are compared with the reference's own output
    (tests/golden/make_golden_big.py), in the benchmark's scan mode and in the reference's default one."""
    g = golden("config2")
    utts = g["utts"].tolist()
    audio = FU.synth_audio(64, 240000).cuda()
    m = make_model(va, mode)
    mel = va.compute_mel_spectrogram(audio)
    assert np.abs(mel[utts][:, ::50].cpu().numpy() - g["mel_sub"]).max() < MEL_ATOL
    logits = m(mel)
    assert logits.shape == (64, 751, 1000)
    ours = logits[utts]
    assert rel(ours[:, ::25], g[mode + "_logits_sub"]) < LOGIT_RTOL
    am = ours.argmax(-1).cpu().numpy()
    # Random-init logits are nearly flat (|logit| <= 2.3, median best-minus-second margin 0.11): 1.1 % of the frames
    # have a margin <= 1e-3 and 0.04 % one <= 1e-5, i.e. inside the reference's own fp32 noise.  A frame counts as
    # decided when its margin exceeds 1e-4 (20x tighter than the 1e-3 logits tolerance would need).
    safe = g[mode + "_margin"] > 1e-4
    assert safe.mean() > 0.99
    assert (am == g[mode + "_argmax"])[safe].all()
    tokens = m.transcribe(audio)                         # the fused call the benchmark times
    assert tokens == va.ctc_greedy_decode(logits)
    pinned = decode_with_reference_on_near_ties(va, ours, g[mode + "_argmax"], safe)
    for row, want in zip(pinned, g[mode + "_tokens"]):
        assert row == [t for t in want.tolist() if t >= 0]
    agree = np.mean([tokens[u] == [t for t in want.tolist() if t >= 0] for u, want in zip(utts, g[mode + "_tokens"])])
    assert agree >= 2 / 3                                # bit-exact unless a near-tie frame flipped


def test_config4_long_form(va, golden):
    """BASELINE configs[3] at reduced batch: one 600 s utterance = 30,001 tokens (1,876 scan chunks of 16 steps,
    K1 = 3,750 pooled tokens, K2 = 64 attention keys), positional table regenerated to 30,008 rows by the
    formula of model.py:94-100, against the reference's own sequential-scan output."""
    g = golden("config4")
    audio = FU.synth_audio(1, 600 * 16000, seed=int(g["seed"])).cuda()
    m = make_model(va, "sequential")
    with pytest.raises(RuntimeError):
        m.transcribe(audio)                              # the stock 5,000-row table is too short (model.py:125)
    m.extend_positional_table(int(g["rows"]))
    mel = va.compute_mel_spectrogram(audio)
    logits, feats = m(mel, return_features=True)
    assert logits.shape == (1, 30001, 1000)
    idx = torch.from_numpy(g["token_idx"]).cuda()
    scale = np.abs(g["local_at"]).max()
    assert np.abs(feats["local_features"][0, idx].cpu().numpy() - g["local_at"]).max() / scale < LOGIT_RTOL
    assert np.abs(feats["local_features"][0, -1].cpu().numpy() - g["local_last"]).max() / scale < LOGIT_RTOL
    assert rel(feats["fused_features"][0, idx], g["fused_at"]) < LOGIT_RTOL
    assert rel(logits[0, idx], g["logits_at"]) < LOGIT_RTOL
    am = logits.argmax(-1).cpu().numpy()
    safe = g["margin"] > 1e-4                            # see test_config2_full_batch
    assert safe.mean() > 0.99
    assert (am == g["argmax"])[safe].all()
    assert decode_with_reference_on_near_ties(va, logits, g["argmax"], safe)[0] == g["tokens"].tolist()
    assert m.transcribe(audio) == va.ctc_greedy_decode(logits)


def test_transcribe_paths_agree_and_shard(va):
    """Fused PCM->tokens == mel + forward + greedy; host-buffer entry == device entry; an
    utterance decodes the same alone as inside a batch (the data-parallel sharding rule)."""
    m = make_model(va, "sequential", amp=True)
    audio = FU.synth_audio(6, 48000, seed=11)
    dev = m.transcribe(audio.cuda())
    host = m.transcribe(audio.pin_memory())
    sep = va.ctc_greedy_decode(m(va.compute_mel_spectrogram(audio.cuda())))
    assert dev == host == sep
    assert m.transcribe(audio[3:5].cuda()) == dev[3:5]
    assert m.transcribe(audio[2].cuda()) == dev[2:3]
    oracle = O.transcribe(audio[:2].numpy(), np_sd(m), dict(scan_mode="sequential"))
    assert oracle == dev[:2]


def test_transcribe_batches_pipeline(va):
    """The pipelined stream API returns exactly what one transcribe() call per batch returns,
    including when the batch shape changes mid-stream."""
    m = make_model(va, "sequential", amp=True)
    batches = [FU.synth_audio(4, 32000, seed=21).pin_memory(), FU.synth_audio(4, 32000, seed=22).pin_memory(),
               FU.synth_audio(2, 48000, seed=23).pin_memory(), FU.synth_audio(4, 32000, seed=24)]
    streamed = list(m.transcribe_batches(iter(batches)))
    assert len(streamed) == len(batches)
    for got, a in zip(streamed, batches):
        assert got == m.transcribe(a.cuda())
    assert list(m.transcribe_batches(iter([]))) == []
    with pytest.raises(RuntimeError):
        list(m.transcribe_batches(iter([batches[0].cuda()])))


def test_transcribe_list_and_trainer_checkpoint(va, tmp_path):
    """f3 / f1 of SURVEY 8f: ragged input without padding; Trainer-format checkpoints (training.py:382-397)."""
    m = make_model(va, "sequential", amp=True)
    lens = [16000, 23456, 16000, 8000, 23456, 16000]
    utts = [FU.synth_audio(1, n, seed=40 + i)[0] for i, n in enumerate(lens)]
    got = m.transcribe_list(utts, max_batch=2)
    assert got == [m.transcribe(u.cuda())[0] for u in utts]
    cfg = va.VelocityASRConfig(scan_mode="sequential", ssm_layers=2, vocab_size=128)
    torch.manual_seed(3)
    small = va.VELOCITYASR(cfg)
    path = str(tmp_path / "trainer.pt")
    torch.save({"model_state_dict": small.state_dict(), "optimizer_state_dict": {}, "scheduler_step": 0,
                "global_step": 7, "best_eval_loss": 1.0, "config": {"learning_rate": 1e-3, "batch_size": 8},
                "model_config": cfg.to_dict()}, path)
    loaded = va.VELOCITYASR.from_pretrained(path).cuda().eval()
    assert loaded.config.ssm_layers == 2 and loaded.config.vocab_size == 128
    mel = va.compute_mel_spectrogram(FU.synth_audio(1, 8000).cuda())
    assert torch.equal(loaded(mel), small.cuda().eval()(mel))


@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_ragged_batch_equals_each_utterance_alone(va, mode):
    """f3 of SURVEY 8f, the masked mode: one padded batch with per-utterance lengths gives every utterance
    bit for bit what it gets alone — logits and tokens — whatever sits in the padding.  Lengths cover every
    branch of the pooling sizes (K1 = L | 64 | L/8, K2 = 16 | K1/4) and odd sample counts."""
    m = make_model(va, mode, amp=True)
    lens = [16000, 4800, 240000, 96000, 23457, 201 + 160, 240000]
    S = max(lens)
    g = torch.Generator().manual_seed(5)
    pcm = torch.randn(len(lens), S, generator=g) * 0.3                 # the padding is noise, not zeros
    for b, n in enumerate(lens):
        pcm[b, :n] = FU.synth_audio(1, n, seed=60 + b)[0]
    alone = [m.transcribe(pcm[b, :n].cuda())[0] for b, n in enumerate(lens)]
    assert m.transcribe(pcm.cuda(), lengths=lens) == alone
    assert m.transcribe(pcm.pin_memory(), lengths=torch.tensor(lens)) == alone      # host entry point
    host = pcm.pin_memory()
    assert list(m.transcribe_batches([(host, lens), host[:2, :16000], (host, lens)])) == \
        [alone, m.transcribe(host[:2, :16000]), alone]                               # pipelined, mixed with plain
    assert any(len(t) > 0 for t in alone)
    # forward with frame counts: logits rows of the valid tokens are identical, padding content is ignored
    mels = [va.compute_mel_spectrogram(pcm[b, :n].cuda()) for b, n in enumerate(lens)]
    T = max(x.shape[0] for x in mels)
    batch = torch.full((len(lens), T, 80), 7.0, device="cuda")
    for b, x in enumerate(mels):
        batch[b, :x.shape[0]] = x
    out = m(batch, lengths=[x.shape[0] for x in mels])
    for b, x in enumerate(mels):
        want = m(x.unsqueeze(0))[0]
        assert torch.equal(out[b, :want.shape[0]], want), (mode, b)
    # full-length utterances in a ragged call are the plain call
    assert torch.equal(m(batch[[2, 6]], lengths=[T, T]), m(batch[[2, 6]]))
    with pytest.raises(RuntimeError):
        m.transcribe(pcm.cuda(), lengths=[200] + lens[1:])
    with pytest.raises(RuntimeError):
        m.transcribe(pcm.cuda(), lengths=[S + 1] + lens[1:])
    with pytest.raises(RuntimeError):
        m.transcribe(pcm.cuda(), lengths=lens[1:])


def test_programmatic_launch_is_a_pure_scheduling_change(va):
    """The kernels of the step are launched with programmatic stream serialisation (common.cuh): the same
    forward in a fresh process with VASR_PDL=0 (plain stream order) must give bit-identical logits."""
    import subprocess
    import sys
    code = (
        "import sys, torch, hashlib; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import fixtures_util as FU, velocity_asr as va\n"
        "torch.manual_seed(FU.WEIGHT_SEED)\n"
        "m = va.VELOCITYASR(va.VelocityASRConfig(scan_mode='sequential')).cuda().eval()\n"
        "out = m(va.compute_mel_spectrogram(FU.synth_audio(3, 24000).cuda()))\n"
        "print(hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest())\n"
    ) % (os.path.join(ROOT, "velocity-asr_b200"), os.path.join(ROOT, "tests"))
    digests = []
    for pdl in ("0", "1"):
        env = dict(os.environ, VASR_PDL=pdl)
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        digests.append(r.stdout.strip().splitlines()[-1])
    assert digests[0] == digests[1]


def test_long_form_needs_longer_table(va):
    m = make_model(va, "sequential")
    mel = torch.randn(1, 10003, 80, device="cuda")      # 5002 tokens > pe_time rows (model.py:87,125)
    with pytest.raises(RuntimeError):
        m(mel)
    m.extend_positional_table(6000)
    out = m(mel)
    assert out.shape == (1, 5002, 1000) and torch.isfinite(out).all()
    sd = np_sd(m)
    ref_tb = O.temporal_binding(mel[:, :400].double().cpu().numpy(), sd)
    _, f = m(mel[:, :400].contiguous(), return_features=True)
    assert rel(f["temporal_binding"], ref_tb) < 1e-4


# ------------------------------------------------------------------ config 5: FakeQuantize ---
def test_quantized_model_matches_reference_golden(va, golden):
    """prepare_model_for_qat + calibrate_model on the CUDA path against the reference run recorded in
    tests/golden/quant.npz (recipe in tests/golden/make_golden_quant.py) and against the oracle."""
    from velocity_asr.quantize import QUANTIZED_MODULES, read_quant_params
    g = golden("quant")
    names = [str(n) for n in g["names"]]
    assert sorted(names) == sorted(QUANTIZED_MODULES)
    m = make_model(va, "sequential")
    mel_cal = va.compute_mel_spectrogram(FU.synth_audio(2, 16000).cuda())
    mel_test = va.compute_mel_spectrogram(FU.synth_audio(2, 16000, seed=77).cuda())
    fp32 = m(mel_test)
    assert rel(fp32, g["logits_fp32"]) < 1e-3
    va.prepare_model_for_qat(m)
    # un-calibrated output nodes pass through (quantize.py:82-84): only the weights are on the int8 grid
    sd = np_sd(m)
    ref_w_only = O.forward(mel_test.double().cpu().numpy(), sd, dict(scan_mode="sequential"), quant=O.QuantState())
    assert rel(m(mel_test), ref_w_only) < 1e-3
    va.calibrate_model(m, [mel_cal])
    got = read_quant_params(m)
    for n, s_ref, z_ref in zip(names, g["act_scale"], g["act_zp"]):
        s_, z_ = got[n]
        assert abs(s_ - s_ref) < 1e-2 * s_ref and abs(z_ - z_ref) < 1.0, (n, s_, s_ref, z_, z_ref)
    step = float(g["act_scale"][names.index("ctc_head.proj.2")])
    # same grids as the reference: load its calibrated parameters, then compare logits
    eng = m._engine(m._device())
    for n, s_ref, z_ref in zip(names, g["act_scale"], g["act_zp"]):
        va._native.check(eng.lib.vasr_set_quant_params(eng.handle, n.encode(), float(s_ref), float(z_ref)))
    lq = m(mel_test).cpu().numpy()
    d = np.abs(lq - g["logits_q"])
    assert (d < 1e-3).mean() > 0.8, (d < 1e-3).mean()
    assert d.max() <= 2.5 * step, (d.max(), step)
    assert (lq.argmax(-1) == g["logits_q"].argmax(-1)).mean() >= 0.95
    # every logit sits on the last quantiser's grid: (x / scale + zp) is an integer in [0, 255]
    s_c, z_c = float(g["act_scale"][names.index("ctc_head.proj.2")]), float(g["act_zp"][names.index("ctc_head.proj.2")])
    qv = lq.astype(np.float64) / s_c + z_c
    assert np.abs(qv - np.rint(qv)).max() < 1e-2 and qv.min() > -0.5 and qv.max() < 255.5
    # tokens: fused path == separate calls, and agree with the reference's argmax stream
    audio = FU.synth_audio(2, 16000, seed=77)
    assert m.transcribe(audio.cuda()) == va.ctc_greedy_decode(m(mel_test))


def test_quantized_modules_one_by_one(va, golden):
    """Each of the 12 quantised modules on its own, fed the INPUT the reference's module saw in its frozen
    forward (tests/golden/quant_modules.npz, forward hooks in make_golden_quant.py) with the reference's
    calibrated scale / zero point: the output must sit on the same grid point everywhere, one quantiser step
    at most where the fp32 value lands within rounding noise of a grid boundary.  This separates "a quantiser
    upstream flipped a step" (what the whole-model test tolerates) from a wrong module."""
    from velocity_asr.quantize import run_quantized_module
    g, gm = golden("quant"), golden("quant_modules")
    names = [str(n) for n in g["names"]]
    m = make_model(va, "sequential")
    va.prepare_model_for_qat(m)
    eng = m._engine(m._device())
    for n, s_ref, z_ref in zip(names, g["act_scale"], g["act_zp"]):
        va._native.check(eng.lib.vasr_set_quant_params(eng.handle, n.encode(), float(s_ref), float(z_ref)))
    m._act_qparams = {n: (float(s_), float(z_)) for n, s_, z_ in zip(names, g["act_scale"], g["act_zp"])}
    site_input = {n: gm[n + ":in"] for n in names}
    # gate_proj.0 / local_proj / global_proj share the projection whose input is [local | ctx]
    cat = np.concatenate([gm["global_context.fusion.local_proj:in"], gm["global_context.fusion.global_proj:in"]], -1)
    assert np.array_equal(cat, gm["global_context.fusion.gate_proj.0:in"])
    for n in ("global_context.fusion.local_proj", "global_context.fusion.global_proj"):
        site_input[n] = cat
    exact_total = 0
    for n, step in zip(names, g["act_scale"]):
        want = gm[n + ":out"]
        got = run_quantized_module(m, n, torch.from_numpy(site_input[n]).cuda()).cpu().numpy()
        assert got.shape == want.shape, n
        d = np.abs(got - want)
        assert d.max() <= 1.001 * step + 1e-6, (n, d.max(), step)
        exact = (d < 1e-3 * step).mean()
        assert exact > 0.995, (n, exact)                     # off-grid-by-one only at boundary ties
        exact_total += exact
    assert exact_total / len(names) > 0.999


def test_quantization_is_reversible_and_guarded(va):
    m = make_model(va, "sequential")
    mel = va.compute_mel_spectrogram(FU.synth_audio(1, 8000).cuda())
    base = m(mel)
    with pytest.raises(RuntimeError):
        va.calibrate_model(m, [mel])                 # prepare_model_for_qat first
    with pytest.raises(NotImplementedError):
        va.prepare_model_for_qat(m, va.QuantizationConfig(weight_bits=4))
    va.prepare_model_for_qat(m)
    va.calibrate_model(m, [mel])
    q = m(mel)
    assert (q - base).abs().max() > 1e-3
    assert torch.equal(m(mel), q)                    # deterministic
    m._quantized = False
    assert torch.equal(m(mel), base)                 # fp32 weights come back bit-identical


# ------------------------------------------------------------------ CTC greedy -----------
def test_ctc_greedy_known_answers(va, golden):
    g = golden("decode")
    for i in range(5):
        lg = torch.nn.functional.one_hot(torch.from_numpy(g[f"in{i}"]).long()[None], 10).float().cuda()
        assert va.ctc_greedy_decode(lg)[0] == g[f"out{i}"].tolist()
        assert va.ctc_greedy_decode(lg, collapse_repeated=False)[0] == g[f"out_nocollapse{i}"].tolist()
    tie = torch.zeros(1, 3, 6); tie[0, 0, 2] = tie[0, 0, 4] = 1.0; tie[0, 1, 5] = 1.0
    assert va.ctc_greedy_decode(tie.cuda())[0] == g["tie_out"].tolist()
    assert va.ctc_greedy_decode(torch.zeros(2, 0, 5).cuda()) == [[], []]
    assert va.ctc_greedy_decode(torch.zeros(0, 4, 5).cuda()) == []
    dec = va.CTCDecoder(va.create_default_vocabulary(10))
    lg = torch.nn.functional.one_hot(torch.tensor([[4, 4, 0, 5, 3, 6]]), 10).float().cuda()
    assert dec.decode_greedy(lg) == ["ab c"]


def test_ctc_timestamps_vs_oracle(va):
    """ctc_greedy_decode_with_timestamps (decode.py:74-125): bit-exact tokens and frame ranges."""
    rs = np.random.RandomState(3)
    # few classes + a strong blank prior -> long runs, repeats across blanks, runs touching both ends
    for (B, L, V) in [(5, 97, 6), (3, 1, 4), (2, 300, 3), (1, 33, 2)]:
        lg = rs.standard_normal((B, L, V)).astype(np.float32)
        lg[..., 0] += 0.8
        lg = np.repeat(lg, 2, axis=1)[:, :L]          # duplicate frames: runs of >= 2
        got = va.ctc_greedy_decode_with_timestamps(torch.from_numpy(lg).cuda())
        assert got == O.ctc_greedy_decode_with_timestamps(lg)
        assert [t for t, _ in got] == va.ctc_greedy_decode(torch.from_numpy(lg).cuda())
    known = np.full((1, 13, 8), -5.0, np.float32)
    for i, t in enumerate([0, 5, 5, 0, 5, 7, 7, 7, 0, 0, 3, 3, 5]):
        known[0, i, t] = 5.0
    assert va.ctc_greedy_decode_with_timestamps(torch.from_numpy(known).cuda()) == \
        [([5, 5, 7, 3, 5], [(1, 3), (4, 5), (5, 8), (10, 12), (12, 13)])]


def test_ctc_beam_search_vs_reference_golden(va, golden):
    """ctc_beam_search (decode.py:128-217) on the device against outputs of the reference itself
    (tests/golden/beam.npz): prefixes, beam order and beam count bit-exact — including the cases whose
    scores tie exactly, where the reference's insertion order decides — and the fp64 scores to the fp32
    rounding of the log-softmax table (1e-4 absolute over <= 40 frames)."""
    g = golden("beam")
    for i in range(int(g["n_cases"])):
        lg, (W, blank) = g[f"lg_{i}"], g[f"par_{i}"].tolist()
        res = va.ctc_beam_search(torch.from_numpy(lg).cuda(), beam_width=W, blank_token=blank)
        want_tok, want_len, want_sc = g[f"tok_{i}"], g[f"len_{i}"], g[f"sc_{i}"]
        for b, beams in enumerate(res):
            assert len(beams) == int((want_len[b] >= 0).sum()), (i, b)
            for r, d in enumerate(beams):
                assert d.tokens == want_tok[b, r, :want_len[b, r]].tolist(), (i, b, r)
                assert abs(d.score - want_sc[b, r]) < 1e-4, (i, b, r)


def test_ctc_beam_search_vs_oracle_and_greedy(va):
    """Larger shapes against the oracle (vocab 1000, the default width 10, 60 frames), and the sanity
    properties: beams are distinct prefixes with non-increasing scores; with peaked frames the best beam is
    the greedy transcript; the decoder class returns texts of the best beam."""
    rs = np.random.RandomState(9)
    lg = (rs.standard_normal((3, 60, 1000)) * 2.5).astype(np.float32)
    res = va.ctc_beam_search(torch.from_numpy(lg).cuda())
    want = O.ctc_beam_search(lg, 10)
    for beams, wb in zip(res, want):
        assert [d.tokens for d in beams] == [t for t, _ in wb]
        assert np.allclose([d.score for d in beams], [s for _, s in wb], rtol=0, atol=2e-4)
        assert len({tuple(d.tokens) for d in beams}) == len(beams) == 10
        assert all(a.score >= b.score for a, b in zip(beams, beams[1:]))
    pred = torch.randint(0, 5, (4, 200), generator=torch.Generator().manual_seed(2))
    pk = (torch.nn.functional.one_hot(pred, 50).float() * 12.0).cuda()
    best = [utt[0].tokens for utt in va.ctc_beam_search(pk, beam_width=4)]
    assert best == va.ctc_greedy_decode(pk)
    dec = va.CTCDecoder(va.create_default_vocabulary(50))
    assert dec.decode_beam_search(pk, beam_width=4) == dec.decode_greedy(pk)
    allb = dec.decode_beam_search(pk, beam_width=3, return_all_beams=True)
    assert len(allb) == 4 and all(len(u) == 3 and isinstance(u[0].text, str) for u in allb)
    assert va.ctc_beam_search(torch.zeros(2, 0, 7).cuda(), 3)[0][0].tokens == []
    with pytest.raises(NotImplementedError):
        va.ctc_beam_search(pk, lm_scorer=object(), lm_weight=0.5)
    with pytest.raises(ValueError):
        va.ctc_beam_search(pk, beam_width=33)


def test_ctc_greedy_random_vs_oracle(va):
    g = torch.Generator().manual_seed(4)
    pred = torch.randint(0, 4, (7, 1003), generator=g)           # many blanks and repeats, ragged outputs
    lg = torch.nn.functional.one_hot(pred, 1000).float() + 0.01 * torch.rand(7, 1003, 1000, generator=g)
    got = va.ctc_greedy_decode(lg.cuda())
    assert got == O.ctc_greedy_decode(lg.numpy())
    assert va.ctc_greedy_decode(lg.cuda(), blank_token=2) == O.ctc_greedy_decode(lg.numpy(), blank_token=2)


def test_non_default_local_stack_config(va):
    """ssm_kernel_size 3, expand_ratio 1, 3 layers of state 32 in the local stack; the global stack keeps the
    reference's hard-coded expand_ratio 2 / kernel_size 4 (ssm.py:529-538).  Against the oracle, both scan modes."""
    for mode in ("sequential", "parallel"):
        torch.manual_seed(21)
        m = va.VELOCITYASR(va.VelocityASRConfig(ssm_layers=3, ssm_state_dim=32, ssm_expand_ratio=1,
                                                ssm_kernel_size=3, scan_mode=mode))
        m.load_state_dict(FU.amplify_state_dict(m.state_dict(), seed=4))
        m = m.cuda().eval()
        audio = FU.synth_audio(2, 12000, seed=8)
        mel = va.compute_mel_spectrogram(audio.cuda())
        got = m(mel)
        want = O.forward(mel.double().cpu().numpy(), np_sd(m),
                         dict(ssm_layers=3, ssm_state_dim=32, ssm_expand_ratio=1, ssm_kernel_size=3, scan_mode=mode))
        assert rel(got, want) < LOGIT_RTOL
        assert m.transcribe(audio.cuda()) == va.ctc_greedy_decode(got)
    with pytest.raises(NotImplementedError):
        va.VELOCITYASR(va.VelocityASRConfig(attention_heads=8, attention_dim=64)).cuda()(mel)   # > 4 heads


@pytest.mark.parametrize("d_model", [96, 128, 160])
def test_other_model_widths(va, d_model):
    """Widths at which the fused epilogues do or do not apply (csrc/engine.cu can_fold_ln, gate_perm_row): 160 folds the
    LayerNorms (five k-blocks) but keeps gate_mix (160 % 64 != 0); 128 keeps the LayerNorm launches, logits and
    argmax_kernel (four k-blocks = the A slots) but mixes the gate in the epilogue; 96 keeps both.  Against the oracle;
    the fused decode must agree with greedy decode of the logits."""
    torch.manual_seed(5)
    cfg = dict(d_model=d_model, ssm_layers=2, global_ssm_layers=1)
    m = va.VELOCITYASR(va.VelocityASRConfig(scan_mode="sequential", **cfg))
    m.load_state_dict(FU.amplify_state_dict(m.state_dict(), seed=6))
    m = m.cuda().eval()
    audio = FU.synth_audio(3, 20000, seed=9)
    mel = va.compute_mel_spectrogram(audio.cuda())
    got = m(mel)
    want = O.forward(mel.double().cpu().numpy(), np_sd(m), dict(scan_mode="sequential", **cfg))
    assert rel(got, want) < LOGIT_RTOL
    assert m.transcribe(audio.cuda()) == va.ctc_greedy_decode(got)
    assert m.transcribe(audio) == va.ctc_greedy_decode(got)            # host entry point


def test_folded_layernorm_survives_a_common_offset(va):
    """LayerNorm folded into the projection (csrc/gemm_tc.cu, EPI_LNA): the row statistics are sums of the row SHIFTED
    by the mean of its first 32 channels, and the shifted row is what the tensor core multiplies — so a common offset
    of the rows (which LayerNorm removes) costs no digits.  Without the shift an offset of 30 standard deviations
    left 2e-4 of the largest logit (E[x^2] - mean^2 cancels as (mean / std)^2)."""
    m = make_model(va, "sequential", amp=True)
    sd = np_sd(m)
    x0 = np.random.RandomState(3).standard_normal((2, 75, 192)).astype(np.float32)
    for c in (0.0, 30.0, 300.0):
        x = (x0 + np.float32(c)).astype(np.float32)
        xt = torch.from_numpy(x).cuda()
        assert rel(m.run_ctc_head(xt), O.ctc_head(x.astype(np.float64), sd)) < 1e-5
        assert rel(m.run_ssm_block(xt, 3, "local"),
                   O.ssm_block(x.astype(np.float64), sd, "local_ssm.layers.3.", "sequential")) < 2e-5


def test_fused_argmax_ties_go_to_the_lowest_index(va):
    """Greedy decode takes the head's per-slot argmax partials (GemmArgs::amax_val): with a zero head weight every
    frame's logits are the bias, so exact ties are under control — inside one 32-column chunk, across the two halves
    of an n-tile and across n-tiles the first maximum must win, as torch.argmax (decode.py:46)."""
    m = make_model(va, "sequential")
    audio = FU.synth_audio(2, 16000, seed=2)
    for hot, want in (((5, 6), 5), ((40, 100), 40), ((130, 700), 130), ((999, 3), 3), ((64, 63), 63)):
        with torch.no_grad():
            m.ctc_head.proj["2"].weight.zero_()
            b = torch.full((1000,), -1.0)
            b[list(hot)] = 2.5
            m.ctc_head.proj["2"].bias.copy_(b)
        m.refresh_weights()
        logits = m(va.compute_mel_spectrogram(audio.cuda()))
        assert int(logits[0, 0].argmax()) == want and float(logits[0, 0].max()) == 2.5
        assert m.transcribe(audio.cuda()) == [[want], [want]]


def test_calls_on_one_handle_are_ordered_across_streams(va):
    """An asynchronous forward on the caller's stream followed at once by a host-tensor transcribe (which runs on the
    handle's own stream) share the workspace: the second call must wait for the first on the device."""
    m = make_model(va, "sequential", amp=True)
    audio = FU.synth_audio(8, 48000, seed=3)
    mel = va.compute_mel_spectrogram(audio.cuda())
    want_logits = m(mel).clone()
    want_tokens = m.transcribe(audio.cuda())
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for _ in range(5):
        with torch.cuda.stream(side):
            logits = m(mel)                        # queued on `side`, not waited for
        tokens = m.transcribe(audio)               # CPU tensor -> the handle's own stream
        side.synchronize()
        assert torch.equal(logits, want_logits)
        assert tokens == want_tokens
    # the device a call runs on is restored afterwards
    assert torch.cuda.current_device() == 0


# ------------------------------------------------------------------ errors ---------------
def test_error_behaviour(va):
    with pytest.raises(ValueError):
        va.VELOCITYASR(va.VelocityASRConfig(scan_mode="bogus"))               # ssm.py:126
    with pytest.raises(ValueError):
        va.selective_scan(*[torch.zeros(1, 1, 64).cuda()] * 2, torch.zeros(64).cuda(),
                          *[torch.zeros(1, 1, 64).cuda()] * 2, scan_mode="bogus")
    with pytest.raises(NotImplementedError):
        va.VELOCITYASR.from_pretrained("velocity-asr-v2-base")                # model.py:409-413
    m = va.VELOCITYASR()
    out = m(torch.zeros(1, 10, 80))            # host model + host input: staged to the GPU, result back on the host
    assert out.device.type == "cpu" and tuple(out.shape) == (1, 5, 1000)
    m = m.cuda()
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 10, 80, device="cuda").to("cuda:0")[:, :, :79].contiguous())   # wrong mel_bins
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 10, 81).cuda())
