"""The greedy path with token timestamps and scores (vasr_ctc_greedy_confidence, vasr_transcribe_timestamps;
include/vasr.h states the rule): ctc_greedy_decode_with_confidence, VELOCITYASR.transcribe_with_timestamps,
words_with_timestamps(..., token_log_probs).

CPU: an fp64 numpy restatement of the rule, pinned on hand-computed cases (a flat row, a tie between blank and a
token, repeats split by a blank, len 0); word confidences; argument checks before any device work, in Python and at
the C ABI.
GPU:
  * from logits: tokens and timestamps equal ctc_greedy_decode_with_timestamps; token and path log-probs within
    1e-5 per frame (+ 1e-6 |ref|) of the oracle; ragged batches with NaN padding equal each utterance alone; the path
    log-prob equals ctc_forced_align's score of the greedy tokens bit for bit and is <= ctc_log_likelihood;
  * fused: tokens equal transcribe() (both scan modes, device and host PCM, ragged or not, FakeQuantize model),
    timestamps equal ctc_greedy_decode_with_timestamps(forward(mel)), scores within the bar of the oracle on
    forward's logits, ragged results equal each utterance alone;
  * the CTC head's softmax-sum epilogue (EPI_ASUM), each of its 4 instantiations through vasr_debug_gemm_asum on two
    shapes or more (one with a partial last m-tile and n-tile), with 1e4-scaled rows, zero rows, flat rows and slots
    past N: val / idx equal the argmax-only instantiation bit for bit, the sums are within 1e-6 relative of fp64
    sum exp(x - v_p) over the output the logits-writing instantiation stores;
  * the merge kernel alone (vasr_debug_confidence) on hand-built partials: empty slots, ties across slots, two slots
    with equal mass, ragged lengths read at a stride, NaN past each length, and log-probs from about -1e-7 to -28, so
    that a path sum added in another order than time order rounds differently.
"""
import ctypes
import math
from ctypes import c_int64, c_void_p

import numpy as np
import pytest
import torch

import fixtures_util as FU
import test_projection_variants as PV

ASUM = 8                      # EPI_ASUM of gemm_tc2_kernel


# ------------------------------------------------------------------ the oracle -----------------------------------
def greedy_oracle(x, n=None, blank=0):
    """The rule in fp64 over the first n rows of x (L, V): (tokens, [(start, end)], token log-probs, path log-prob)."""
    x = np.asarray(x, np.float64)
    n = x.shape[0] if n is None else n
    x = x[:n]
    if n == 0:
        return [], [], [], 0.0
    a = x.argmax(axis=1)
    m = x.max(axis=1)
    lp = x[np.arange(n), a] - (m + np.log(np.exp(x - m[:, None]).sum(axis=1)))
    tokens, spans, tlps = [], [], []
    t = 0
    while t < n:
        if a[t] == blank:
            t += 1
            continue
        s = t
        while t < n and a[t] == a[s]:
            t += 1
        tokens.append(int(a[s]))
        spans.append((s, t))
        tlps.append(float(lp[s:t].sum()))
    return tokens, spans, tlps, float(lp.sum())


def test_oracle_flat_row():
    V = 5
    assert greedy_oracle(np.zeros((1, V)), blank=3) == ([0], [(0, 1)], [pytest.approx(-math.log(V), abs=1e-15)],
                                                         pytest.approx(-math.log(V), abs=1e-15))
    assert greedy_oracle(np.zeros((1, V)), blank=0) == ([], [], [], pytest.approx(-math.log(V), abs=1e-15))


def test_oracle_tie_between_blank_and_token():
    tok, spans, tlps, lp = greedy_oracle([[2.0, 2.0, 0.0]], blank=0)           # the blank is the lower index
    assert (tok, spans, tlps) == ([], [], [])
    assert lp == pytest.approx(2.0 - math.log(2 * math.exp(2.0) + 1.0), abs=1e-15)
    tok, spans, tlps, _ = greedy_oracle([[0.0, 2.0, 2.0]], blank=2)             # the token is the lower index
    assert (tok, spans) == ([1], [(0, 1)])


def test_oracle_repeats_split_by_a_blank():
    l3 = math.log(3.0)
    x = [[0, l3, 0], [0, l3, 0], [l3, 0, 0], [0, l3, 0], [0, 0, l3], [0, 0, l3]]    # argmax 1 1 0 1 2 2
    tok, spans, tlps, lp = greedy_oracle(x, blank=0)
    per = l3 - math.log(5.0)                                                    # every frame: 3 / (3 + 1 + 1)
    assert tok == [1, 1, 2] and spans == [(0, 2), (3, 4), (4, 6)]
    assert tlps == [pytest.approx(2 * per, abs=1e-15), pytest.approx(per, abs=1e-15), pytest.approx(2 * per, abs=1e-15)]
    assert lp == pytest.approx(6 * per, abs=1e-14)                              # blank frames count in the path


def test_oracle_len_zero():
    assert greedy_oracle(np.ones((4, 3)), 0) == ([], [], [], 0.0)


def test_word_confidence():
    import velocity_asr as va
    vocab = ["_", " ", "a", "b"]
    tokens, stamps = [2, 3, 1, 2], [(0, 2), (3, 4), (4, 5), (6, 9)]
    plain = va.words_with_timestamps(tokens, stamps, vocab)
    assert all("confidence" not in w for w in plain)
    tlp = [-0.2, -0.4, -5.0, -0.9]
    words = va.words_with_timestamps(tokens, stamps, vocab, token_log_probs=tlp)
    assert [{k: w[k] for k in ("word", "start", "end")} for w in words] == plain
    assert words[0]["confidence"] == pytest.approx(math.exp((-0.2 - 0.4) / 3))     # the separator is excluded
    assert words[1]["confidence"] == pytest.approx(math.exp(-0.9 / 3))


def test_checks_before_device_work():
    import velocity_asr as va
    x = torch.zeros(2, 5, 4)
    with pytest.raises(RuntimeError):
        va.ctc_greedy_decode_with_confidence(x, lengths=[5, 6])
    with pytest.raises(RuntimeError):
        va.ctc_greedy_decode_with_confidence(x, lengths=[5])
    with pytest.raises(ValueError):
        va.ctc_greedy_decode_with_confidence(x, blank_token=4)


def test_c_abi_checks_before_device_work():
    from velocity_asr import _native
    lib = _native.lib()
    host = np.zeros(16, np.float64)             # any non-null address: the checks fail before it is touched
    p = lambda a: c_void_p(a.ctypes.data)
    rows = np.array([3, 6], np.int32)
    code = lib.vasr_ctc_greedy_confidence(p(host), p(rows), 2, 5, 4, 0, p(host), p(host), p(host), p(host), p(host),
                                          p(host), None)
    assert code == _native.ERR_SHAPE
    code = lib.vasr_ctc_greedy_confidence(p(host), None, 2, 5, 4, 4, p(host), p(host), p(host), p(host), p(host),
                                          p(host), None)
    assert code == _native.ERR_INVALID
    code = lib.vasr_ctc_greedy_confidence(p(host), None, 2, 5, 4, 0, p(host), p(host), p(host), p(host), None,
                                          p(host), None)
    assert code == _native.ERR_INVALID
    code = lib.vasr_ctc_greedy_confidence(p(host), None, -1, 5, 4, 0, p(host), p(host), p(host), p(host), p(host),
                                          p(host), None)
    assert code == _native.ERR_SHAPE


# ------------------------------------------------------------------ GPU: from logits -----------------------------
@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


def check_result(r, want, frames, what):
    tokens, spans, tlps, lp = want
    assert r.tokens == tokens and r.timestamps == spans, what
    for k, (s, e) in enumerate(spans):
        assert abs(r.token_log_probs[k] - tlps[k]) <= 1e-5 * (e - s) + 1e-6 * abs(tlps[k]), (what, k)
    assert abs(r.log_prob - lp) <= 1e-5 * frames + 1e-6 * abs(lp), what


def random_logits(seed, B, L, V, scale=2.5, blank_bias=1.5):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, L, V, generator=g) * scale
    x[..., 0] += blank_bias                    # blank-heavy, as a CTC head is: runs, blank frames and repeats
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("V", [40, 1000])
def test_from_logits(va, V):
    B, L = 6, 300
    x = random_logits(V, B, L, V)
    res = va.ctc_greedy_decode_with_confidence(x.cuda())
    ts = va.ctc_greedy_decode_with_timestamps(x.cuda())
    for b in range(B):
        assert (res[b].tokens, res[b].timestamps) == (ts[b][0], ts[b][1]), b
        check_result(res[b], greedy_oracle(x[b].numpy()), L, f"utterance {b}")
    assert sum(len(r.tokens) for r in res) > 10 * B
    # the path log-prob is the forced alignment's score of the greedy tokens: the same fp32 table, fp64 time order
    al = va.ctc_forced_align(x.cuda(), [r.tokens for r in res])
    ll = va.ctc_log_likelihood(x.cuda(), [r.tokens for r in res]).cpu().tolist()
    for b in range(B):
        assert res[b].log_prob == al[b].score, b
        assert res[b].log_prob <= ll[b], b
        flp = al[b].frame_log_probs.double().numpy()
        for k, (s, e) in enumerate(res[b].timestamps):     # fp64 time-order sums of the same fp32 values
            acc = 0.0
            for t in range(s, e):
                acc += float(flp[t])
            assert res[b].token_log_probs[k] == acc, (b, k)


@pytest.mark.gpu
def test_from_logits_ragged_equals_alone(va):
    B, L, V = 7, 200, 96
    x = random_logits(3, B, L, V)
    lens = [200, 0, 1, 57, 199, 128, 3]
    xp = x.clone()
    for b, n in enumerate(lens):
        xp[b, n:] = float("nan")                           # padding is never read
    res = va.ctc_greedy_decode_with_confidence(xp.cuda(), lengths=lens)
    for b, n in enumerate(lens):
        alone = va.ctc_greedy_decode_with_confidence(x[b:b + 1, :n].cuda())[0]
        assert res[b] == alone, b
        check_result(res[b], greedy_oracle(x[b].numpy(), n), n, f"utterance {b}")
    assert res[1].tokens == [] and res[1].log_prob == 0.0
    host = va.ctc_greedy_decode_with_confidence(xp, lengths=torch.tensor(lens))       # host logits are staged
    assert host == res


# ------------------------------------------------------------------ GPU: fused --------------------------------------
SAMPLE_LENS = [16000, 4800, 240000, 96000, 23457, 201 + 160]


def make_model(va, mode):
    torch.manual_seed(FU.WEIGHT_SEED)
    m = va.VELOCITYASR(va.VelocityASRConfig(scan_mode=mode))
    m.load_state_dict(FU.amplify_state_dict(m.state_dict()))
    return m.cuda().eval()


def padded_pcm():
    S = max(SAMPLE_LENS)
    g = torch.Generator().manual_seed(5)
    pcm = torch.randn(len(SAMPLE_LENS), S, generator=g) * 0.3
    for b, n in enumerate(SAMPLE_LENS):
        pcm[b, :n] = FU.synth_audio(1, n, seed=60 + b)[0]
    return pcm


def check_fused(va, m, exact_scores):
    """exact_scores: the fused call takes the from-logits route (FakeQuantize model), so its scores are
    ctc_greedy_decode_with_confidence's on forward's logits bit for bit."""
    pcm = padded_pcm()
    res = m.transcribe_with_timestamps(pcm.cuda(), lengths=SAMPLE_LENS)
    assert m.transcribe_with_timestamps(pcm, lengths=torch.tensor(SAMPLE_LENS)) == res        # host PCM
    assert [r.tokens for r in res] == m.transcribe(pcm.cuda(), lengths=SAMPLE_LENS)
    for b, n in enumerate(SAMPLE_LENS):
        one = pcm[b:b + 1, :n]
        alone = m.transcribe_with_timestamps(one.cuda())[0]
        assert res[b] == alone, b
        assert alone.tokens == m.transcribe(one.cuda())[0]
        logits = m(va.compute_mel_spectrogram(one.cuda()))
        tokens, stamps = va.ctc_greedy_decode_with_timestamps(logits)[0]
        assert (alone.tokens, alone.timestamps) == (tokens, stamps), b
        check_result(alone, greedy_oracle(logits[0].cpu().numpy()), logits.shape[1], f"utterance {b}")
        if exact_scores:
            assert alone == va.ctc_greedy_decode_with_confidence(logits)[0], b
    assert sum(len(r.tokens) for r in res) > 0
    same = torch.stack([pcm[2], pcm[2]])                   # not ragged
    both = m.transcribe_with_timestamps(same.cuda())
    assert both[0] == both[1] == m.transcribe_with_timestamps(same[:1])[0] == res[2]
    assert [r.tokens for r in both] == m.transcribe(same.cuda())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_fused_equals_transcribe_and_forward(va, mode):
    check_fused(va, make_model(va, mode), exact_scores=False)


@pytest.mark.gpu
def test_fused_quantized_model(va):
    m = make_model(va, "sequential")
    va.prepare_model_for_qat(m)
    va.calibrate_model(m, [va.compute_mel_spectrogram(FU.synth_audio(2, 16000).cuda())])
    check_fused(va, m, exact_scores=True)


@pytest.mark.gpu
def test_fused_errors(va):
    m = make_model(va, "sequential")
    pcm = FU.synth_audio(2, 8000).cuda()
    with pytest.raises(RuntimeError):
        m.transcribe_with_timestamps(pcm[:, :150])                      # too short for the reflect padding
    with pytest.raises(RuntimeError):
        m.transcribe_with_timestamps(pcm, lengths=[8000, 9000])          # longer than S
    assert m.transcribe_with_timestamps(pcm[:0]) == []


# ------------------------------------------------------------------ GPU: the softmax-sum epilogue ----------------
def _asum_cases():
    C = []
    for wr, shapes in ((1, [(1000, 60, 192, 2), (12016, 1000, 192, 0)]), (0, [(257, 1000, 384, 0), (255, 60, 192, 0)])):
        for M, N, K, sms in shapes:
            C.append(PV.Case(PV._v(2, 128, PV.NONE, wr=wr, epi=PV.LNA | PV.AMAX | ASUM), M, N, K, ln_offset=30.0,
                             amax=True, num_sms=sms, seed=70 + len(C)))
    for wr, shapes in ((1, [(1000, 60, 4, 2), (2000, 400, 96, 16)]), (0, [(257, 1000, 240, 0), (31, 60, 36, 0),
                                                                          (129, 132, 4, 0)])):
        for M, N, K, sms in shapes:
            C.append(PV.Case(PV._v(2, 128, PV.NONE, wr=wr, epi=PV.AMAX | ASUM), M, N, K, amax=True, num_sms=sms,
                             seed=70 + len(C)))
    return C


ASUM_CASES = _asum_cases()


def asum_id(c):
    return PV.vname(c.expect[:7] + (c.expect[7] & ~ASUM,)) + f"-asum-M{c.M}-N{c.N}-K{c.K}"


def test_asum_cases_cover_each_instantiation_with_a_ragged_shape():
    kinds = {c.expect for c in ASUM_CASES}
    assert len(kinds) == 4
    for v in kinds:
        cs = [c for c in ASUM_CASES if c.expect == v]
        assert len({(c.M, c.N, c.K) for c in cs}) >= 2
        assert any(c.M % 256 and c.N % 128 for c in cs), v


@pytest.fixture(scope="module")
def asum_seam():
    from velocity_asr import _native
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    fn = _native.lib().vasr_debug_gemm_asum
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.POINTER(PV._GemmCall), c_void_p]
    plain = _native.lib().vasr_debug_gemm
    plain.restype = ctypes.c_int
    plain.argtypes = [ctypes.POINTER(PV._GemmCall)]
    return fn, plain


def run_asum(asum_seam, p):
    """(variant, val, idx, sum) with the softmax-sum epilogue, the (val, idx) of the argmax-only instantiation and
    the output of the logits-writing one, for the same inputs."""
    fn, plain = asum_seam
    c = p.c
    slots = 2 * ((c.N + 127) // 128)
    sums = torch.full((slots * c.M + 64,), float(PV.SENTINEL), device="cuda")
    rc, v, _, av, ai = p.run(lambda g: fn(g, c_void_p(sums.data_ptr())))
    assert rc == 0, "vasr_debug_gemm_asum"
    rc, v1, _, av1, ai1 = p.run(plain)
    assert rc == 0 and v1[7] == c.expect[7] & ~ASUM
    rc, v2, Cbuf, _, _ = p.run(plain, amax=False)
    assert rc == 0 and not v2[7] & PV.AMAX
    s = sums.cpu().numpy()
    assert (s[slots * c.M:] == PV.SENTINEL).all(), "wrote past the slots"
    assert av.tobytes() == av1.tobytes() and ai.tobytes() == ai1.tobytes(), "val / idx differ from the AMAX variant"
    return v, av[:slots * c.M].reshape(slots, c.M), ai[:slots * c.M].reshape(slots, c.M), \
        s[:slots * c.M].reshape(slots, c.M), Cbuf[:c.M, :c.N]


def check_sums(val, sums, out, N, what):
    slots = val.shape[0]
    for q in range(slots):
        lo, hi = 64 * q, min(64 * q + 64, N)
        if lo >= hi:
            assert (sums[q] == 0).all(), f"{what}: empty slot {q}"
            continue
        ref = np.exp(out[:, lo:hi].astype(np.float64) - val[q].astype(np.float64)[:, None]).sum(axis=1)
        err = np.abs(sums[q] - ref) / ref
        assert err.max() <= 1e-6, f"{what}: slot {q} rel err {err.max():.2e} at row {err.argmax()}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", ASUM_CASES, ids=[asum_id(c) for c in ASUM_CASES])
def test_asum_epilogue(asum_seam, case):
    p = PV.Problem(case)
    v, val, idx, sums, out = run_asum(asum_seam, p)
    assert v == case.expect
    assert (np.abs(p.A).max(axis=1) > 1e3).any()           # 1e4-scaled rows are in the batch
    check_sums(val, sums, out, case.N, asum_id(case))


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in ASUM_CASES if c.M % 256 and c.N % 128],
                         ids=[asum_id(c) for c in ASUM_CASES if c.M % 256 and c.N % 128])
def test_asum_zero_and_flat_rows(asum_seam, case):
    """Zero bias (and beta): the zero rows of A give x = 0 in every column, so each slot's sum is its column count
    exactly.  Then zero weights: every row is flat."""
    p = PV.Problem(case)
    p.b[:] = 0.0
    if p.ln is not None:
        p.ln = (p.ln[0], np.zeros_like(p.ln[1]), p.ln[2])
    _, val, _, sums, out = run_asum(asum_seam, p)
    zero = np.flatnonzero(np.abs(p.A).max(axis=1) == 0)
    assert zero.size
    counts = np.array([max(min(64 * q + 64, case.N) - 64 * q, 0) for q in range(val.shape[0])], np.float32)
    assert (sums[:, zero] == counts[:, None]).all()
    check_sums(val, sums, out, case.N, "zero bias")
    p = PV.Problem(case)
    p.W[:] = 0.0
    p.b[:] = 3.0
    if p.ln is not None:
        p.ln = (p.ln[0], np.zeros_like(p.ln[1]), p.ln[2])
    _, val, idx, sums, out = run_asum(asum_seam, p)
    assert (sums == counts[:, None]).all()
    live = counts > 0
    assert (idx[live] == (64 * np.arange(val.shape[0]))[live][:, None]).all()


# ------------------------------------------------------------------ GPU: the merge kernel alone ------------------
class _ConfCall(ctypes.Structure):
    _fields_ = [("logits", c_void_p), ("stats", c_void_p), ("V", c_int64),
                ("amax_val", c_void_p), ("amax_idx", c_void_p), ("amax_sum", c_void_p), ("slots", c_int64),
                ("pred", c_void_p), ("lp", c_void_p),
                ("tokens", c_void_p), ("starts", c_void_p), ("ends", c_void_p), ("token_log_probs", c_void_p),
                ("lens", c_void_p), ("log_probs", c_void_p),
                ("lens_in", c_void_p), ("lens_stride", c_int64),
                ("B", c_int64), ("L", c_int64), ("blank", c_int64), ("stream", c_void_p)]


def hand_partials(rs, B, L, slots):
    """Slot partials (val, idx, sum) as the head leaves them, with the special frames named in the docstring."""
    val = (rs.standard_normal((slots, B, L)) * 3).astype(np.float32)
    idx = (64 * np.arange(slots)[:, None, None] + rs.randint(0, 64, size=(slots, B, L))).astype(np.int32)
    val[:, :, 0::3] += np.float32(4.0) * (idx[:, :, 0::3] < 64)          # blank-heavy frames keep runs short
    idx[0, :, 0::3] = 0
    sm = rs.uniform(1.0, 64.0, size=(slots, B, L)).astype(np.float32)
    # t = 1: the last two slots are empty (a vocabulary of 128 or fewer columns)
    val[2:, :, 1], idx[2:, :, 1], sm[2:, :, 1] = -np.inf, -1, 0.0
    # t = 2: slots 1 and 2 tie for the maximum: slot 1 wins
    val[1, :, 2] = val[2, :, 2] = val[:, :, 2].max(axis=0) + 1
    # t = 4: slots 0 and 3 carry equal mass at different maxima (sum_0 e^v0 == sum_3 e^v3)
    val[0, :, 4], sm[0, :, 4] = 2.0, np.float32(8.0)
    val[3, :, 4], sm[3, :, 4] = 1.0, np.float32(8.0 * math.e)
    val[1:3, :, 4] = -3.0
    # t = 8, 13, 18, ...: confident frames, Z = 1 + O(1e-7) and lp_t of about -1e-7 among frames of about -3: an fp64
    # sum of the fp32 lp_t then rounds, so the order of the path's sum shows in its bits
    conf = np.sort(np.concatenate([np.arange(8, L, 5), np.arange(10, L, 5)]))
    val[0, :, conf], sm[0, :, conf], idx[0, :, conf] = 10.0, 1.0, 5
    val[1:, :, conf] = (10.0 - rs.uniform(16.2, 17.5, size=(slots - 1, B, conf.size))).astype(np.float32)
    sm[1:, :, conf] = 1.0
    # t = 6, 11, 16, ...: unlikely frames, lp_t of about -28, so the path's sum runs to about -2e3 while the confident
    # frames add bits 60 octaves below its leading one
    sm[:, :, np.arange(6, L, 5)] = 1e12
    return val, idx, sm


def merge_oracle(val, idx, sm):
    """Per frame: the prediction (slot order, a later slot on a strictly greater value) and -log Z in fp64."""
    slots = val.shape[0]
    best = np.full(val.shape[1:], -np.inf)
    bi = np.full(val.shape[1:], -1)
    for q in range(slots):
        take = (idx[q] >= 0) & ((val[q] > best) | (bi < 0))
        best = np.where(take, val[q], best)
        bi = np.where(take, idx[q], bi)
    z = np.zeros(val.shape[1:])
    for q in range(slots):
        z += np.where(idx[q] >= 0, sm[q].astype(np.float64) * np.exp(val[q].astype(np.float64) - best), 0.0)
    return bi, -np.log(z)


@pytest.mark.gpu
def test_merge_kernel_on_hand_built_partials(va):
    from velocity_asr import _native
    fn = _native.lib().vasr_debug_confidence
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.POINTER(_ConfCall)]
    rs = np.random.RandomState(11)
    B, L, slots, blank = 8, 300, 4, 0
    val, idx, sm = hand_partials(rs, B, L, slots)
    lens = [300, 0, 5, 211, 300, 280, 250, 299]
    want_pred, want_lp = merge_oracle(val, idx, sm)
    assert (want_pred[:, 2] == idx[1, :, 2]).all()
    nan_val, nan_idx, nan_sm = val.copy(), idx.copy(), sm.copy()
    for b, n in enumerate(lens):                        # never read: NaN values, indices that would win
        nan_val[:, b, n:], nan_idx[:, b, n:], nan_sm[:, b, n:] = np.nan, 7, np.nan
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    dv, di, ds = d(nan_val.reshape(slots, -1)), d(nan_idx.reshape(slots, -1)), d(nan_sm.reshape(slots, -1))
    lens_in = d(np.array([[n, -5] for n in lens], np.int32))           # read at a stride of 2
    pred = torch.full((B, L), -7, dtype=torch.int32, device="cuda")
    lp = torch.full((B, L), 99.0, device="cuda")
    outs = [torch.full((B, L), -9, dtype=torch.int32, device="cuda") for _ in range(3)]
    tlp = torch.full((B, L), 99.0, dtype=torch.float64, device="cuda")
    olens = torch.full((B,), -9, dtype=torch.int32, device="cuda")
    plp = torch.full((B,), 99.0, dtype=torch.float64, device="cuda")
    a = _ConfCall(amax_val=dv.data_ptr(), amax_idx=di.data_ptr(), amax_sum=ds.data_ptr(), slots=slots,
                  pred=pred.data_ptr(), lp=lp.data_ptr(), tokens=outs[0].data_ptr(), starts=outs[1].data_ptr(),
                  ends=outs[2].data_ptr(), token_log_probs=tlp.data_ptr(), lens=olens.data_ptr(),
                  log_probs=plp.data_ptr(), lens_in=lens_in.data_ptr(), lens_stride=2, B=B, L=L, blank=blank,
                  stream=torch.cuda.current_stream().cuda_stream)
    assert fn(ctypes.byref(a)) == 0
    pred, lp, tlp, plp = pred.cpu().numpy(), lp.cpu().numpy(), tlp.cpu().numpy(), plp.cpu().numpy()
    tok, st, en = (o.cpu().numpy() for o in outs)
    olens = olens.cpu().tolist()
    for b, n in enumerate(lens):
        assert (pred[b, :n] == want_pred[b, :n]).all(), b
        assert (pred[b, n:] == -7).all() and (lp[b, n:] == 99.0).all(), f"{b}: wrote past the length"
        err = np.abs(lp[b, :n] - want_lp[b, :n])
        assert (err <= 2e-6 * np.maximum(1.0, np.abs(want_lp[b, :n]))).all(), (b, err.max())
        # runs of the merged predictions, and fp64 time-order sums of the kernel's own fp32 lp
        x = np.full((n, 2 ** 8), 0.0)
        x[np.arange(n), pred[b, :n]] = 1.0
        tokens, spans, _, _ = greedy_oracle(x, n, blank)
        assert olens[b] == len(tokens)
        assert tok[b, :olens[b]].tolist() == tokens and list(zip(st[b, :olens[b]].tolist(),
                                                                 en[b, :olens[b]].tolist())) == spans
        assert (tok[b, olens[b]:] == -1).all() and (tlp[b, olens[b]:] == 0).all()
        for k, (s, e) in enumerate(spans):
            acc = 0.0
            for t in range(s, e):
                acc += float(lp[b, t])
            assert tlp[b, k] == acc, (b, k)
        acc = 0.0
        for t in range(n):
            acc += float(lp[b, t])
        assert plp[b] == acc, b
    rev = []
    for b, n in enumerate(lens):
        acc = 0.0
        for t in reversed(range(n)):
            acc += float(lp[b, t])
        rev.append(acc)
    assert (np.array(rev) != plp).any(), "the inputs do not make the order of the path's sum visible"
    assert olens[1] == 0 and plp[1] == 0.0
    # t = 4: Z = 8 e^0 + 8e e^(1 - 2) + (sum_1 + sum_2) e^(-3 - 2), each slot rescaled to the frame's maximum
    z = 16.0 + (float(sm[1, 0, 4]) + float(sm[2, 0, 4])) * math.exp(-5.0)
    assert want_lp[0, 4] == pytest.approx(-math.log(z), rel=1e-7)
