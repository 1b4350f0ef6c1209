"""CTC forced alignment and transcript log-likelihood on the device (vasr_ctc_align, vasr_ctc_log_likelihood,
vasr_align; include/vasr.h states the rule).

CPU: the numpy oracle (align_oracle.py) against torch's ctc_loss, against brute-force enumeration of every
alignment (score, the path the tie rule names, log-add), and against torchaudio's forced_align where ties cannot
occur; malformed ids and lengths are refused before any device work, in Python and at the C ABI.
GPU: with log_probs=True the device equals the oracle bit for bit (labels, frame log-probs, fp64 scores) over
continuous, coarse-grid and all-tied tables; raw logits; consistency with the greedy decode and the beam search;
ragged batches against each utterance alone; long targets (both score layouts); the fused PCM path; CTCDecoder.align.
"""
import ctypes
import itertools
import math
import warnings

import numpy as np
import pytest
import torch

import align_oracle as AO
import fixtures_util as FU


def random_target(rs, U, V, blank=0, repeat_p=0.3):
    """U ids in [0, V) without the blank; a token repeats its predecessor with probability repeat_p (always when
    there is a single non-blank id), never otherwise."""
    ids = [i for i in range(V) if i != blank]
    y = []
    for _ in range(U):
        if y and (rs.rand() < repeat_p or len(ids) == 1):
            y.append(y[-1])
        else:
            others = [i for i in ids if not y or i != y[-1]]
            y.append(others[rs.randint(len(others))])
    return y


def repeats(y):
    return sum(1 for a, b in zip(y[:-1], y[1:]) if a == b)


def log_softmax32(x):
    return torch.log_softmax(torch.from_numpy(np.asarray(x, np.float32)), dim=-1).numpy()


# ------------------------------------------------------------------ CPU: the oracle -------------------------------
def ctc_loss64(lp, y, blank=0):
    """torch's CTC loss (fp64, reduction none) of one utterance."""
    lp_t = torch.from_numpy(np.asarray(lp, np.float64)).unsqueeze(1)        # (T, 1, V)
    tgt = torch.tensor([y if y else [1]], dtype=torch.long)
    return float(torch.nn.functional.ctc_loss(lp_t, tgt, torch.tensor([lp_t.shape[0]]), torch.tensor([len(y)]),
                                              blank=blank, reduction="none", zero_infinity=False)[0])


@pytest.mark.parametrize("seed", range(6))
def test_oracle_log_likelihood_equals_ctc_loss(seed):
    rs = np.random.RandomState(seed)
    V = 7
    cases = []
    for _ in range(8):                                     # random targets with repeats
        U = rs.randint(1, 9)
        y = random_target(rs, U, V)
        cases.append((rs.randint(U + repeats(y), 30), y))
    cases.append((12, []))                                 # U = 0: the all-blank path
    y = random_target(rs, 6, V, repeat_p=0.6)
    cases.append((len(y) + repeats(y), y))                 # tight: T = U + repeats
    cases.append((len(y) + repeats(y) - 1, y))             # one frame short: cannot fit
    cases.append((3, [1, 1, 1]))                           # 3 < 3 + 2
    for T, y in cases:
        lp = np.log(rs.dirichlet(np.ones(V), size=T))
        want = -ctc_loss64(lp, y)
        got = AO.log_likelihood(lp, y)
        if math.isinf(want):
            assert got == -math.inf, (T, y)
        else:
            assert got == pytest.approx(want, rel=1e-9, abs=0), (T, y)


def enumerate_paths(lp, y, blank=0):
    """Every alignment of y over lp's frames: (state path, time-ordered fp64 score)."""
    T, V = lp.shape
    out = []
    for pi in itertools.product(range(V), repeat=T):
        coll, prev = [], None
        states, k = [], 0
        for p in pi:
            if p != blank and p != prev:
                coll.append(p)
            prev = p
        if coll != list(y):
            continue
        prev = None
        for p in pi:                                        # blank before token k -> 2k, token k -> 2k + 1
            if p == blank:
                states.append(2 * k)
            else:
                if p != prev:
                    k += 1
                states.append(2 * k - 1)
            prev = p
        score = 0.0
        for t, p in enumerate(pi):
            score += float(lp[t, p])
        out.append((states, score))
    return out


def rule_path(paths, U):
    """The path the tie rule names among the best: the last-token final state over the trailing blank, then,
    frame by frame backwards, the highest predecessor state (stay before s-1 before s-2)."""
    best = max(s for _, s in paths)
    top = [p for p, s in paths if s == best]
    return max(top, key=lambda p: ((p[-1] == 2 * U - 1),) + tuple(reversed(p[:-1])))


TINY = [(t, u, v) for t in (1, 2, 3, 5, 8) for u in (0, 1, 2, 3) for v in (2, 3, 4)
        if u <= t and not (t == 8 and v == 4 and u != 3)]     # 4^8 paths: one case there keeps the run short


@pytest.mark.parametrize("grid", ["continuous", "coarse", "tied"])
@pytest.mark.parametrize("T,U,V", TINY)
def test_oracle_against_enumeration(T, U, V, grid):
    rs = np.random.RandomState(T * 100 + U * 10 + V)
    if grid == "continuous":
        lp = log_softmax32(rs.standard_normal((T, V)) * 2)
    elif grid == "coarse":                                  # a few exactly representable values: many exact ties
        lp = (-0.5 * rs.randint(0, 3, size=(T, V))).astype(np.float32)
    else:
        lp = np.full((T, V), -math.log(V), np.float32)
    for y in (random_target(rs, U, V, repeat_p=0.5), random_target(rs, U, V, repeat_p=0.0)):
        labels, flp, score = AO.viterbi(lp, y)
        paths = enumerate_paths(lp, y)
        if not paths:
            assert score == -math.inf and (labels == -1).all() and (flp == 0).all()
            assert AO.log_likelihood(lp, y) == -math.inf
            continue
        assert score == max(s for _, s in paths)
        lab, _ = AO.lattice(y, 0)
        want = rule_path(paths, len(y))
        assert labels.tolist() == [int(lab[s]) for s in want], (lp.tolist(), y)
        assert flp.tolist() == [float(lp[t, lab[s]]) for t, s in enumerate(want)]
        m = max(s for _, s in paths)
        ll = m + math.log(sum(math.exp(s - m) for _, s in paths))
        assert AO.log_likelihood(lp, y) == pytest.approx(ll, rel=1e-12, abs=1e-12)


@pytest.mark.parametrize("seed", range(10))
def test_oracle_path_equals_torchaudio_on_continuous_inputs(seed):
    F = pytest.importorskip("torchaudio.functional")
    rs = np.random.RandomState(seed)
    V = 12
    for _ in range(10):
        U = rs.randint(1, 20)
        y = random_target(rs, U, V)
        T = rs.randint(U + repeats(y), 3 * U + 10)
        lp = np.log(rs.dirichlet(np.ones(V) * 0.5, size=T))  # fp64, continuous: no ties
        labels, _, score = AO.viterbi(lp, y)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")                 # torchaudio's deprecation notice
            ta, _ = F.forced_align(torch.from_numpy(lp).unsqueeze(0), torch.tensor([y], dtype=torch.int32), blank=0)
        assert labels.tolist() == ta[0].tolist(), (seed, y)


# ------------------------------------------------------------------ CPU: argument checks -------------------------
def test_malformed_ids_and_lengths_raise_before_device_work():
    import velocity_asr as va
    lg = torch.zeros(2, 5, 4)                       # host logits: a device call would come after the checks
    for fn in (va.ctc_forced_align, va.ctc_log_likelihood):
        with pytest.raises(ValueError, match="outside"):
            fn(lg, [[1, 0], [2]])                   # the blank
        with pytest.raises(ValueError, match="outside"):
            fn(lg, [[1], [4]])                      # id >= V
        with pytest.raises(ValueError, match="outside"):
            fn(lg, [[-1], [2]])
        with pytest.raises(ValueError, match="blank token"):
            fn(lg, [[1], [2]], blank_token=4)
        with pytest.raises(RuntimeError, match="expected 2 targets"):
            fn(lg, [[1]])
        with pytest.raises(RuntimeError, match="expected 2 lengths"):
            fn(lg, [[1], [2]], lengths=[3])
        with pytest.raises(RuntimeError, match=r"in \[0, 5\]"):
            fn(lg, [[1], [2]], lengths=[3, 6])
        with pytest.raises(RuntimeError, match=r"in \[0, 5\]"):
            fn(lg, [[1], [2]], lengths=torch.tensor([-1, 2]))
    with pytest.raises(RuntimeError, match="expected 2 targets"):
        va.CTCDecoder(["<blank>", "a", "b", "c"]).align(lg, ["ab"])


def _abi_args(targets, tlens, rows, U_max, B=2, L=5, V=4):
    host = np.zeros((B, L, V), np.float32)
    tg = np.asarray(targets, np.int32).reshape(B, max(U_max, 1))
    return host, tg, np.asarray(tlens, np.int32), None if rows is None else np.asarray(rows, np.int32)


@pytest.mark.parametrize("case,exc,msg", [
    (dict(targets=[[1, 0], [2, 3]], tlens=[2, 2], rows=None, U_max=2), ValueError, "outside the vocabulary"),
    (dict(targets=[[1, 4], [2, 3]], tlens=[2, 2], rows=None, U_max=2), ValueError, "outside the vocabulary"),
    (dict(targets=[[1, 2], [2, 3]], tlens=[3, 2], rows=None, U_max=2), RuntimeError, r"\[0, U_max\]"),
    (dict(targets=[[1, 2], [2, 3]], tlens=[-1, 2], rows=None, U_max=2), RuntimeError, r"\[0, U_max\]"),
    (dict(targets=[[1, 2], [2, 3]], tlens=[2, 2], rows=[6, 2], U_max=2), RuntimeError, "between 0 and L"),
    (dict(targets=[[1, 2], [2, 3]], tlens=[2, 2], rows=[-1, 2], U_max=2), RuntimeError, "between 0 and L"),
    # only the first target_lens[b] ids of a row are read: the blank past it is no error, the length is
    (dict(targets=[[1, 0], [2, 3]], tlens=[1, 2], rows=[6, 2], U_max=2), RuntimeError, "between 0 and L"),
])
def test_c_abi_checks_before_device_work(case, exc, msg):
    """vasr_ctc_align / vasr_ctc_log_likelihood refuse bad ids (VASR_ERR_INVALID) and lengths (VASR_ERR_SHAPE) with
    host arrays only: the checks come before any device call."""
    from velocity_asr import _native
    host, tg, tl, rows = _abi_args(**case)
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    out_i = np.zeros(16, np.int32)
    out_f = np.zeros(16, np.float32)
    out_d = np.zeros(4, np.float64)
    lib = _native.lib()
    with pytest.raises(exc, match=msg):
        _native.check(lib.vasr_ctc_align(p(host), p(rows), 2, 5, 4, 0, 0, p(tg), p(tl), case["U_max"], p(out_i),
                                         p(out_f), p(out_d), None))
    with pytest.raises(exc, match=msg):
        _native.check(lib.vasr_ctc_log_likelihood(p(host), p(rows), 2, 5, 4, 0, 1, p(tg), p(tl), case["U_max"],
                                                  p(out_d), None))


def test_c_abi_checks_blank_and_null_pointers():
    from velocity_asr import _native
    host, tg, tl, _ = _abi_args([[1, 2], [2, 3]], [2, 2], None, 2)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    out_i, out_f, out_d = np.zeros(16, np.int32), np.zeros(16, np.float32), np.zeros(4, np.float64)
    lib = _native.lib()
    with pytest.raises(ValueError, match="blank"):
        _native.check(lib.vasr_ctc_align(p(host), None, 2, 5, 4, 4, 0, p(tg), p(tl), 2, p(out_i), p(out_f), p(out_d),
                                         None))
    with pytest.raises(ValueError, match="null"):
        _native.check(lib.vasr_ctc_align(p(host), None, 2, 5, 4, 0, 0, None, p(tl), 2, p(out_i), p(out_f), p(out_d),
                                         None))
    with pytest.raises(ValueError, match="null"):
        _native.check(lib.vasr_ctc_log_likelihood(p(host), None, 2, 5, 4, 0, 0, p(tg), p(tl), 2, None, None))


# ------------------------------------------------------------------ GPU ------------------------------------------
@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


def lp_table(rs, T, V, grid):
    if grid == "continuous":
        return log_softmax32(rs.standard_normal((T, V)) * 2.5)
    if grid == "coarse":
        return (-0.25 * rs.randint(0, 4, size=(T, V))).astype(np.float32)
    return np.full((T, V), -math.log(V), np.float32)


def batch_cases(rs, L, V):
    """(row_len, target) pairs covering U = 0, L = 0, repeats, tight, infeasible and U = L."""
    cases = [(L, []), (0, []), (0, [1]), (1, [2]), (L, random_target(rs, L // 3, V)),
             (L, random_target(rs, L // 2, V, repeat_p=0.5))]
    y = random_target(rs, L // 2, V, repeat_p=0.4)
    cases += [(len(y) + repeats(y), y), (len(y) + repeats(y) - 1, y)]            # tight, one frame short
    y = random_target(rs, L, V, repeat_p=0.0)
    cases += [(L, y), (L - 1, y)]                                                # U = L, and one frame short
    while len(cases) < 64:
        n = int(rs.randint(0, L + 1))
        U = int(rs.randint(0, n + 1))
        cases.append((n, random_target(rs, U, V, repeat_p=rs.choice([0.0, 0.3, 0.9]))))
    return cases


def run_oracle(lp, n, y):
    return AO.viterbi(lp[:n], y) + (AO.log_likelihood(lp[:n], y),)


def assert_exact(res, ll, want, what):
    for b, (labels, flp, score, want_ll) in enumerate(want):
        r = res[b]
        assert r.frame_labels.tolist() == labels.tolist(), (what, b)
        assert r.frame_log_probs.numpy().tobytes() == flp.astype(np.float32).tobytes(), (what, b)
        assert r.score == score, (what, b)
        assert (r.timestamps is None) == (score == -math.inf), (what, b)
        if r.timestamps is not None:
            assert r.timestamps == AO.spans(labels), (what, b)
        got = float(ll[b])
        if want_ll == -math.inf:
            assert got == -math.inf, (what, b)
        else:
            assert got == pytest.approx(want_ll, rel=1e-12, abs=0), (what, b)


@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["continuous", "coarse", "tied"])
@pytest.mark.parametrize("V", [40, 1000])
def test_log_probs_equal_oracle(va, V, grid):
    rs = np.random.RandomState(V + len(grid))
    L = 60
    cases = batch_cases(rs, L, V)
    lp = np.stack([lp_table(rs, L, V, grid) for _ in cases])
    rows = [n for n, _ in cases]
    for b, n in enumerate(rows):
        lp[b, n:] = np.nan
    targets = [y for _, y in cases]
    x = torch.from_numpy(lp).cuda()
    res = va.ctc_forced_align(x, targets, lengths=rows, log_probs=True)
    ll = va.ctc_log_likelihood(x, targets, lengths=rows, log_probs=True).cpu()
    assert ll.dtype == torch.float64 and ll.shape == (len(cases),)
    assert_exact(res, ll, [run_oracle(lp[b], n, y) for b, (n, y) in enumerate(cases)], (V, grid))
    assert any(r.score == -math.inf for r in res) and any(len(r.tokens) == L for r in res if r.timestamps)
    # the whole batch with L = 0
    empty = torch.zeros(3, 0, V, device="cuda")
    res0 = va.ctc_forced_align(empty, [[], [1], []], log_probs=True)
    assert [r.score for r in res0] == [0.0, -math.inf, 0.0]
    assert [r.timestamps for r in res0] == [[], None, []]
    assert va.ctc_log_likelihood(empty, [[], [1], []], log_probs=True).tolist() == [0.0, -math.inf, 0.0]


@pytest.mark.gpu
@pytest.mark.parametrize("V", [40, 1000])
def test_raw_logits_match_oracle_on_torch_log_softmax(va, V):
    rs = np.random.RandomState(7 + V)
    B, L = 16, 120
    lg = (rs.standard_normal((B, L, V)) * 3).astype(np.float32)
    targets = [random_target(rs, int(rs.randint(0, L // 2)), V) for _ in range(B)]
    res = va.ctc_forced_align(torch.from_numpy(lg).cuda(), targets)
    ll = va.ctc_log_likelihood(torch.from_numpy(lg).cuda(), targets).cpu()
    lp = log_softmax32(lg)
    for b, y in enumerate(targets):
        labels, _, score = AO.viterbi(lp[b], y)
        assert res[b].frame_labels.tolist() == labels.tolist(), b
        assert res[b].score == pytest.approx(score, abs=2e-4, rel=0)
        assert float(ll[b]) == pytest.approx(AO.log_likelihood(lp[b], y), abs=2e-4, rel=0)
    # host logits are staged to the device
    host = va.ctc_forced_align(torch.from_numpy(lg[:2]), targets[:2])
    assert [r.frame_labels.tolist() for r in host] == [r.frame_labels.tolist() for r in res[:2]]
    assert va.ctc_log_likelihood(torch.from_numpy(lg[:2]), targets[:2]).device.type == "cpu"


@pytest.mark.gpu
def test_greedy_tokens_align_to_the_argmax_path(va):
    rs = np.random.RandomState(3)
    B, L, V = 32, 200, 50
    lg = (rs.standard_normal((B, L, V)) * 2).astype(np.float32)
    lg[:, :, 0] += 1.5                                        # plenty of blanks, as in real CTC output
    top2 = np.sort(lg, axis=-1)[..., -2:]
    am = lg.argmax(-1)[..., None]                             # widen every frame's top-2 margin to >= 1e-3
    bump = np.where(top2[..., 1] - top2[..., 0] < 1e-2, np.float32(1e-2), np.float32(0))[..., None]
    np.put_along_axis(lg, am, np.take_along_axis(lg, am, -1) + bump, -1)
    top2 = np.sort(lg, axis=-1)[..., -2:]
    assert (top2[..., 1] - top2[..., 0] >= 1e-3).all()
    x = torch.from_numpy(lg).cuda()
    greedy = va.ctc_greedy_decode_with_timestamps(x)
    res = va.ctc_forced_align(x, [g[0] for g in greedy])
    argmax = lg.argmax(-1)
    for b, (toks, spans) in enumerate(greedy):
        assert res[b].frame_labels.tolist() == argmax[b].tolist(), b
        assert res[b].timestamps == spans, b


@pytest.mark.gpu
def test_beam_scores_never_exceed_the_alignment(va):
    rs = np.random.RandomState(5)
    B, L, V = 8, 100, 40
    x = torch.from_numpy((rs.standard_normal((B, L, V)) * 2).astype(np.float32)).cuda()
    beams = va.ctc_beam_search(x, beam_width=10)
    for b, utt in enumerate(beams):
        res = va.ctc_forced_align(x[b:b + 1].expand(len(utt), L, V), [d.tokens for d in utt])
        for d, r in zip(utt, res):
            assert r.score >= d.score, (b, d.tokens)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [40, 1000])
def test_ragged_equals_each_utterance_alone(va, V):
    rs = np.random.RandomState(11 + V)
    B, L = 10, 80
    lg = (rs.standard_normal((B, L, V)) * 2).astype(np.float32)
    rows = [0, 1, L] + [int(n) for n in rs.randint(2, L, size=B - 3)]
    for b, n in enumerate(rows):
        lg[b, n:] = np.nan
    targets = [random_target(rs, int(rs.randint(0, max(n // 2, 1))), V) for n in rows]
    targets[0], targets[1] = [], [3]
    x = torch.from_numpy(lg).cuda()
    for log_probs in (False, True):
        got = va.ctc_forced_align(x, targets, lengths=rows, log_probs=log_probs)
        ll = va.ctc_log_likelihood(x, targets, lengths=rows, log_probs=log_probs).cpu()
        for b, n in enumerate(rows):
            alone = va.ctc_forced_align(x[b:b + 1, :n], targets[b:b + 1], log_probs=log_probs)[0]
            assert got[b].frame_labels.tolist() == alone.frame_labels.tolist(), b
            assert got[b].frame_log_probs.numpy().tobytes() == alone.frame_log_probs.numpy().tobytes(), b
            assert got[b].score == alone.score and got[b].timestamps == alone.timestamps, b
            one = va.ctc_log_likelihood(x[b:b + 1, :n], targets[b:b + 1], log_probs=log_probs)
            assert float(ll[b]) == float(one[0]) or (math.isnan(float(ll[b])) and math.isnan(float(one[0]))), b
        assert got[0].score == 0.0 and got[0].timestamps == [] and got[1].timestamps == [(0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("L,U", [(30001, 9000), (16000, 14000)])
def test_long_targets_against_oracle(va, L, U):
    """U = 9,000 keeps the state scores in shared memory; U = 14,000 (29,001 states) does not fit there and runs the
    global-memory layout, both for the alignment and the log-likelihood."""
    rs = np.random.RandomState(L + U)
    V, B = 40, 2 if U < 12000 else 1                      # the oracle takes about 20 s per utterance here
    lp = np.stack([log_softmax32(rs.standard_normal((L, V)) * 2) for _ in range(B)])
    targets = [random_target(rs, U - 17 * b, V, repeat_p=0.05) for b in range(B)]
    x = torch.from_numpy(lp).cuda()
    res = va.ctc_forced_align(x, targets, log_probs=True)
    ll = va.ctc_log_likelihood(x, targets, log_probs=True).cpu()
    assert_exact(res, ll, [run_oracle(lp[b], L, y) for b, y in enumerate(targets)], (L, U))
    assert all(r.timestamps is not None for r in res)


SAMPLE_LENS = [16000, 4800, 240000, 96000, 23457, 201 + 160, 240000]


def make_model(va, mode):
    torch.manual_seed(FU.WEIGHT_SEED)
    m = va.VELOCITYASR(va.VelocityASRConfig(scan_mode=mode))
    m.load_state_dict(FU.amplify_state_dict(m.state_dict()))
    return m.cuda().eval()


def padded_pcm():
    S = max(SAMPLE_LENS)
    g = torch.Generator().manual_seed(5)
    pcm = torch.randn(len(SAMPLE_LENS), S, generator=g) * 0.3             # the padding is noise, not zeros
    for b, n in enumerate(SAMPLE_LENS):
        pcm[b, :n] = FU.synth_audio(1, n, seed=60 + b)[0]
    return pcm


def fused_targets(m, V):
    rs = np.random.RandomState(9)
    out = []
    for b, n in enumerate(SAMPLE_LENS):
        Lb = m.get_output_length(1 + n // 160)
        out.append(random_target(rs, max(Lb // 4, 1), V))
    out[1] = []                                                              # U = 0
    out[5] = random_target(rs, m.get_output_length(1 + SAMPLE_LENS[5] // 160) + 1, V)   # cannot fit
    return out


def results_of(res):
    return [(r.frame_labels.tolist(), r.frame_log_probs.numpy().tobytes(), r.score, r.timestamps) for r in res]


def assert_fused_equals_composed(va, m):
    V = m.config.vocab_size
    pcm = padded_pcm()
    targets = fused_targets(m, V)
    want = []
    for b, n in enumerate(SAMPLE_LENS):
        logits = m(va.compute_mel_spectrogram(pcm[b, :n].cuda()).unsqueeze(0))
        want += results_of(va.ctc_forced_align(logits, targets[b:b + 1]))
    assert want[5][2] == -math.inf and want[0][2] > -math.inf
    assert results_of(m.align(pcm.cuda(), targets, lengths=SAMPLE_LENS)) == want
    assert results_of(m.align(pcm, targets, lengths=torch.tensor(SAMPLE_LENS))) == want      # host PCM
    full = [2, 6]
    assert results_of(m.align(pcm[full].cuda(), [targets[b] for b in full])) == [want[b] for b in full]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["sequential", "parallel"])
def test_fused_align_equals_composed(va, mode):
    assert_fused_equals_composed(va, make_model(va, mode))


@pytest.mark.gpu
def test_fused_align_quantized_model(va):
    m = make_model(va, "sequential")
    va.prepare_model_for_qat(m)
    va.calibrate_model(m, [va.compute_mel_spectrogram(FU.synth_audio(2, 16000).cuda())])
    assert_fused_equals_composed(va, m)


@pytest.mark.gpu
def test_fused_align_errors(va):
    m = make_model(va, "sequential")
    pcm = FU.synth_audio(2, 8000).cuda()
    with pytest.raises(ValueError):
        m.align(pcm, [[1], [0]])
    with pytest.raises(ValueError):
        m.align(pcm, [[1], [m.config.vocab_size]])
    with pytest.raises(RuntimeError):
        m.align(pcm, [[1]])
    with pytest.raises(RuntimeError):
        m.align(pcm, [[1], [2]], lengths=[8000])
    with pytest.raises(RuntimeError):
        m.align(pcm, [[1], [2]], lengths=[8000, 200])                        # too short for the mel


@pytest.mark.gpu
def test_decoder_align_gives_the_greedy_words(va):
    vocab = ["<blank>", " "] + list("abcdefgh")
    dec = va.CTCDecoder(vocab)
    texts = ["ab ba cab", "hedge", "a agh"]
    L, V = 64, len(vocab)
    lg = np.zeros((len(texts), L, V), np.float32)
    for b, text in enumerate(texts):
        path = [0, 0, 0]
        for ch in text:
            path += [vocab.index(ch)] * 2 + [0]
        path += [0] * (L - len(path))
        lg[b, np.arange(L), path] = 5.0
        lg[b] += np.random.RandomState(b).uniform(0, 0.5, size=(L, V)).astype(np.float32)
    x = torch.from_numpy(lg).cuda()
    greedy = dec.decode_greedy(x)
    assert greedy == texts
    stamps = va.ctc_greedy_decode_with_timestamps(x)
    want = [va.words_with_timestamps(t, s, vocab) for t, s in stamps]
    assert dec.align(x, greedy) == want
    assert all(len(w) > 0 for w in want)
