"""The streaming kernels of the step one launcher at a time, against fp64 references built from the numpy oracle.

The projections have their own file (test_projection_variants.py).  The other kernels of a step, LayerNorm, the
LayerNorm + causal depthwise conv prologue of an SSM block, adaptive pooling, the attention core, the gate mix, the
greedy decode and the FakeQuantize calibration, are reached through the debug seam `vasr_debug_kernel`
(csrc/engine.cu). It calls the real launcher of kernels.cuh with every argument exposed. The log-mel front end is
checked through the public `compute_mel_spectrogram(n_mels=...)`.

What each comparison asserts:
  * float kernels: per output row, max |got - ref| <= bar * max |ref row|.  Bars, and in brackets the worst row
    measured on a B200 (1000 W limit) as a fraction of its bar:
      layer_norm 2e-6 x (1 + |row mean| / row std)   [0.08: 2.3e-5 on a 300-sigma row, whose fp32 mean costs digits]
      ln_dwconv  the same, over the k rows an output reads   [0.14: 4.6e-5 on a 500-sigma row]
      adaptive_pool 1e-6   [0.28]
      attention  2e-6 x max(1, max |score|)   [0.005: 6.8e-6 with scores around 1e3]
      gate_mix   1e-6   [0.14]
    The bars sit far below every mutation the suite is meant to see: LayerNorm eps 1e-6 instead of 1e-5 moves a row
    of variance 1e-4 by 4.5e-2 of its scale, a pooling window one row short moves a mean by about 1/9.
  * log-mel: max-abs error <= 1e-4, the project's mel bar (test_gpu_parity).  Measured 9.4e-5 (n_mels 90, white
    noise): the fp32 FFT's error in the weakest bins, which have the smallest filter weights, after the normalisation
    scales it by 1 / std.
The file takes about 6 s on a B200.
  * integer kernels (decode, timestamps) and the FakeQuantize parameters: bit for bit.
  * NaN in every gap of a strided input and past each ragged utterance's end, a sentinel around every output: a
    kernel that reads outside its input, or writes outside its output, fails.

VASR_ERR_LOG=<file> appends the worst error of each float comparison to that file, for re-deriving the bars.
"""
import ctypes
import os
from ctypes import c_char_p, c_int32, c_int64, c_void_p

import numpy as np
import pytest

import velocity_oracle as O

pytestmark = pytest.mark.gpu

SENT = -7777.25                       # float sentinel around outputs
ISENT = -7                            # int sentinel
RAG_S, RAG_T, RAG_L, RAG_K1, RAG_K2, RAG_STRIDE = 0, 1, 2, 3, 4, 8     # columns of the ragged dims (kernels.cuh)
OK, ERR_UNSUPPORTED = 0, 5

RTOL_LN = 2e-6
RTOL_DW = 2e-6
RTOL_POOL = 1e-6
RTOL_ATT = 2e-6
RTOL_MIX = 1e-6
MEL_ATOL = 1e-4


class _Args(ctypes.Structure):
    _fields_ = [("kernel", c_char_p), ("x", c_void_p), ("ldx", c_int64), ("kv", c_void_p), ("y", c_void_p),
                ("ldy", c_int64), ("gamma", c_void_p), ("beta", c_void_p), ("w", c_void_p), ("bias", c_void_p),
                ("pred", c_void_p), ("tokens", c_void_p), ("lens", c_void_p), ("starts", c_void_p), ("ends", c_void_p),
                ("amax_val", c_void_p), ("amax_idx", c_void_p), ("slots", c_int32),
                ("mm", c_void_p), ("q_scale", c_void_p), ("q_zp", c_void_p), ("c0", c_int32), ("nc", c_int32),
                ("rag", c_void_p), ("f_in", c_int32), ("f_out", c_int32),
                ("B", c_int64), ("L", c_int64), ("M", c_int64), ("K", c_int64),
                ("C", c_int32), ("k", c_int32), ("heads", c_int32), ("hd", c_int32), ("V", c_int32),
                ("blank", c_int32), ("collapse", c_int32), ("run_len", c_int32),
                ("stream", c_void_p), ("run_len_used", c_int32)]


@pytest.fixture(scope="module")
def torch():
    import torch as t
    assert t.cuda.is_available(), "GPU tests need a CUDA device"
    return t


@pytest.fixture(scope="module")
def seam(torch):
    from velocity_asr import _native
    fn = _native.lib().vasr_debug_kernel
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.POINTER(_Args)]

    def call(kernel, **kw):
        a = _Args()
        a.kernel = kernel.encode()
        for k, v in kw.items():
            setattr(a, k, v.data_ptr() if hasattr(v, "data_ptr") else v)
        a.stream = torch.cuda.current_stream().cuda_stream
        rc = fn(ctypes.byref(a))
        return rc, a
    return call


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rag_dims(torch, B, **cols):
    """(B, RAG_STRIDE) int32 on the device; cols: column index -> per-utterance values."""
    r = np.zeros((B, RAG_STRIDE), np.int32)
    for col, vals in cols.items():
        r[:, globals()[col]] = vals
    return dev(torch, r)


def check_rows(name, got, ref, bar):
    """got, ref (R, n); bar: scalar or (R,) relative to each row's max |ref|."""
    got = np.asarray(got, np.float64)
    assert np.isfinite(got).all(), f"{name}: non-finite output"
    scale = np.maximum(np.abs(ref).max(axis=1), 1e-30)
    err = np.abs(got - ref).max(axis=1) / scale
    rel = err / bar
    log = os.environ.get("VASR_ERR_LOG")
    if log:
        with open(log, "a") as f:
            f.write(f"{name}\t{err.max():.3e}\t{rel.max():.3f}\n")
    worst = int(np.argmax(rel))
    assert rel.max() <= 1.0, f"{name}: row {worst} error {err[worst]:.3e} > bar {np.broadcast_to(bar, err.shape)[worst]:.1e}"


# ------------------------------------------------------------------ layer_norm -------------------
def ln_rows(rng, M, C):
    """Rows of N(0, 1), then special rows: 300 sigma offset, constant, scaled by 1e4, variance 1e-4."""
    x = rng.standard_normal((M, C)).astype(np.float32)
    x[1::7] += np.float32(300.0)
    x[2::7] = np.float32(3.0)                      # constant: exact mean, variance 0 -> rstd = 1 / sqrt(eps)
    x[3::7] *= np.float32(1e4)
    x[4::7] *= np.float32(1e-2)                   # variance 1e-4: eps is 10% of it
    return x


def ln_bar(x):
    x = x.astype(np.float64)
    sd = x.std(axis=1)
    return RTOL_LN * (1.0 + np.abs(x.mean(axis=1)) / np.maximum(sd, 1e-30) * (sd > 0))


@pytest.mark.parametrize("C", [64, 96, 128, 160, 192, 200, 256])
@pytest.mark.parametrize("layout", ["dense", "strided", "inplace"])
def test_layer_norm(torch, seam, C, layout):
    M = 203                                        # not a multiple of the 8 rows of a CTA
    rng = np.random.default_rng(C)
    x = ln_rows(rng, M, C)
    g = (1.0 + 0.3 * rng.standard_normal(C)).astype(np.float32)
    b = (0.3 * rng.standard_normal(C)).astype(np.float32)
    ref = O.layer_norm(x.astype(np.float64), g.astype(np.float64), b.astype(np.float64))
    ld = 2 * C if layout == "strided" else C
    store = np.full((M + 1, ld), np.nan, np.float32)
    store[:M, :C] = x
    xs = dev(torch, store)
    if layout == "inplace":
        ys, ldy = xs, ld
    else:
        ldy = C + 3
        ys = torch.full((M + 2, ldy), SENT, device="cuda")
    rc, _ = seam("layer_norm", x=xs, ldx=ld, y=ys, ldy=ldy, gamma=dev(torch, g), beta=dev(torch, b), M=M, C=C)
    assert rc == OK
    out = ys.cpu().numpy()
    check_rows(f"layer_norm C{C} {layout}", out[:M, :C], ref, ln_bar(x))
    assert (out[2:M:7, :C] == b).all()             # constant rows: exactly beta
    if layout == "inplace":
        assert np.isnan(out[:M, C:]).all() and np.isnan(out[M:]).all()
    else:
        assert (out[:M, C:] == SENT).all() and (out[M:] == SENT).all()


def test_layer_norm_declines_257_channels(torch, seam):
    x = torch.zeros(8, 257, device="cuda")
    rc, _ = seam("layer_norm", x=x, ldx=257, y=x, ldy=257, gamma=x, beta=x, M=8, C=257)
    assert rc == ERR_UNSUPPORTED


# ------------------------------------------------------------------ ln_dwconv --------------------
def dw_inputs(rng, B, L, C, K):
    x = rng.standard_normal((B, L, C)).astype(np.float32)
    x[:, 3::5] *= np.float32(1e-2)                # variance 1e-4 rows: the eps shows
    x[:, 4::11] += np.float32(5.0)
    g = (1.0 + 0.3 * rng.standard_normal(C)).astype(np.float32)
    b = (0.3 * rng.standard_normal(C)).astype(np.float32)
    w = (rng.standard_normal((C, K)) / np.sqrt(K)).astype(np.float32)
    bias = rng.standard_normal(C).astype(np.float32)
    return x, g, b, w, bias


def dw_reference(x, g, b, w, bias):
    d = lambda a: a.astype(np.float64)
    u = O.layer_norm(d(x), d(g), d(b))
    return O.causal_depthwise_conv(u, d(w)[:, None, :], d(bias))


def dw_bar(x, K):
    """ln_bar of the K input rows each output row reads (a row far off zero costs its LayerNorm digits)."""
    B, L, C = x.shape
    f = (ln_bar(x.reshape(-1, C)) / RTOL_LN).reshape(B, L)
    f = np.concatenate([np.ones((B, K - 1)), f], axis=1)
    return RTOL_DW * np.lib.stride_tricks.sliding_window_view(f, K, axis=1).max(axis=2).reshape(-1)


def run_dw(torch, seam, x, g, b, w, bias, run_len):
    B, L, C = x.shape
    K = w.shape[1]
    u = torch.full((B * L + 4, C), SENT, device="cuda")
    rc, a = seam("ln_dwconv", x=dev(torch, x), y=u, gamma=dev(torch, g), beta=dev(torch, b), w=dev(torch, w),
                 bias=dev(torch, bias), B=B, L=L, C=C, k=K, run_len=run_len)
    assert rc == OK
    out = u.cpu().numpy()
    assert (out[B * L:] == SENT).all()
    return out[:B * L].reshape(B, L, C), a.run_len_used


@pytest.mark.parametrize("K", range(1, 9))
@pytest.mark.parametrize("C", [64, 96, 160, 192])
def test_ln_dwconv(torch, seam, K, C):
    """L in {1, K-1, K, 751} in one batch each; forced run lengths 4, 5, 16, 64 and the launcher's rule give the same
    bits, including run_len < K - 1 where a run's halo spans earlier runs."""
    rng = np.random.default_rng(10 * K + C)
    for L in sorted({1, max(K - 1, 1), K, 751}):
        x, g, b, w, bias = dw_inputs(rng, 2, L, C, K)
        ref = dw_reference(x, g, b, w, bias)
        first = None
        for run_len in (0, 4, 5, 16, 64):
            out, used = run_dw(torch, seam, x, g, b, w, bias, run_len)
            assert used == run_len or (run_len == 0 and 4 <= used <= 64)
            if first is None:
                check_rows(f"ln_dwconv K{K} C{C} L{L}", out.reshape(-1, C), ref.reshape(-1, C), dw_bar(x, K))
                first = out
            else:
                assert np.array_equal(out, first), f"run_len {run_len} changed the result (K{K} C{C} L{L})"


def test_ln_dwconv_long_and_zero_padding(torch, seam):
    """A long utterance, and the zero left padding: the first K - 1 outputs of utterance 1 must not see the
    last rows of utterance 0, whatever those hold."""
    rng = np.random.default_rng(7)
    K, C, L = 4, 192, 30001
    x, g, b, w, bias = dw_inputs(rng, 2, L, C, K)
    ref = dw_reference(x, g, b, w, bias)
    out, _ = run_dw(torch, seam, x, g, b, w, bias, 0)
    check_rows("ln_dwconv long", out.reshape(-1, C), ref.reshape(-1, C), dw_bar(x, K))
    x2 = x.copy()
    x2[0, -K:] *= np.float32(1e3)
    x2[0, -K:] += np.float32(50.0)
    out2, _ = run_dw(torch, seam, x2, g, b, w, bias, 5)
    assert np.array_equal(out2[1], out[1])


def test_ln_dwconv_declines(torch, seam):
    x = torch.zeros(64, 224, device="cuda")
    rc, _ = seam("ln_dwconv", x=x, y=x, gamma=x, beta=x, w=x, bias=x, B=1, L=4, C=224, k=4)
    assert rc == ERR_UNSUPPORTED
    rc, _ = seam("ln_dwconv", x=x, y=x, gamma=x, beta=x, w=x, bias=x, B=1, L=4, C=64, k=9)
    assert rc == ERR_UNSUPPORTED


# ------------------------------------------------------------------ adaptive_pool ----------------
@pytest.mark.parametrize("L,K,C", [(100, 7, 64), (64, 64, 96), (50, 1, 192), (751, 93, 192), (30001, 3750, 64),
                                   (5, 3, 200), (3, 5, 64)])
@pytest.mark.parametrize("strided", [False, True])
def test_adaptive_pool(torch, seam, L, K, C, strided):
    rng = np.random.default_rng(L + K)
    B = 2
    x = rng.standard_normal((B, L, C)).astype(np.float32)
    ld = 2 * C if strided else C
    store = np.full((B * L, ld), np.nan, np.float32)
    store[:, :C] = x.reshape(B * L, C)
    out = torch.full((B * K + 3, C), SENT, device="cuda")
    rc, _ = seam("adaptive_pool", x=dev(torch, store), ldx=ld, y=out, B=B, L=L, K=K, C=C)
    assert rc == OK
    got = out.cpu().numpy()
    ref = O.adaptive_avg_pool(x.astype(np.float64), K).reshape(B * K, C)
    check_rows(f"adaptive_pool L{L} K{K} C{C}", got[:B * K], ref, RTOL_POOL)
    assert (got[B * K:] == SENT).all()


def test_adaptive_pool_ragged(torch, seam):
    """Each utterance pools its own Lb rows into its own Kb rows (the pool sizes of the model); the rows past Kb
    are zeroed, and the rows past Lb, NaN here, are never read."""
    rng = np.random.default_rng(3)
    L, C = 751, 192
    Ls = [751, 500, 129, 64, 63]
    Ks = [O.pool_sizes(l)[0] for l in Ls]
    B, K = len(Ls), max(Ks)
    x = np.full((B, L, C), np.nan, np.float32)
    for i, l in enumerate(Ls):
        x[i, :l] = rng.standard_normal((l, C))
    rag = rag_dims(torch, B, RAG_L=Ls, RAG_K1=Ks)
    out = torch.full((B * K + 3, C), SENT, device="cuda")
    rc, _ = seam("adaptive_pool", x=dev(torch, x), ldx=C, y=out, B=B, L=L, K=K, C=C, rag=rag, f_in=RAG_L,
                 f_out=RAG_K1)
    assert rc == OK
    got = out.cpu().numpy()
    for i, (l, k) in enumerate(zip(Ls, Ks)):
        rows = got[i * K:(i + 1) * K]
        check_rows(f"adaptive_pool ragged L{l}", rows[:k], O.adaptive_avg_pool(x[i:i + 1, :l].astype(np.float64), k)[0],
                   RTOL_POOL)
        assert (rows[k:] == 0).all()
    assert (got[B * K:] == SENT).all()


# ------------------------------------------------------------------ attention --------------------
def att_reference(q, k, v, heads):
    """softmax(q k^T / sqrt(hd)) v per head, as in O.multi_head_attention; q (L, A), k / v (Kk, A)."""
    L, A = q.shape
    hd = A // heads
    qh = q.reshape(L, heads, hd).transpose(1, 0, 2)
    kh = k.reshape(-1, heads, hd).transpose(1, 0, 2)
    vh = v.reshape(-1, heads, hd).transpose(1, 0, 2)
    s = qh @ kh.transpose(0, 2, 1) / np.sqrt(hd)
    smax = np.abs(s).max(axis=(0, 2))
    s = s - s.max(axis=-1, keepdims=True)
    p = np.exp(s)
    p = p / p.sum(axis=-1, keepdims=True)
    return (p @ vh).transpose(1, 0, 2).reshape(L, A), smax


def run_attention(torch, seam, q, kv, heads, hd, Kk, Ks=None, scale=1.0):
    """q (B, L, A), kv (B, Kk, 2A); Ks: per-utterance key counts (ragged).  q and o rows are strided (NaN / sentinel
    in the gaps)."""
    B, L, A = q.shape
    ldq, ldo = A + 4, A + 8
    qs = np.full((B * L, ldq), np.nan, np.float32)
    qs[:, :A] = q.reshape(B * L, A)
    o = torch.full((B * L + 2, ldo), SENT, device="cuda")
    rag = rag_dims(torch, B, RAG_K2=Ks) if Ks is not None else None
    kw = dict(rag=rag) if rag is not None else {}
    rc, _ = seam("attention", x=dev(torch, qs), ldx=ldq, kv=dev(torch, kv.reshape(B * Kk, 2 * A)), y=o, ldy=ldo,
                 B=B, L=L, K=Kk, heads=heads, hd=hd, **kw)
    assert rc == OK
    got = o.cpu().numpy()
    assert (got[:B * L, A:] == SENT).all() and (got[B * L:] == SENT).all()
    for b in range(B):
        kb = Kk if Ks is None else Ks[b]
        k = kv[b, :kb, :A].astype(np.float64)
        v = kv[b, :kb, A:].astype(np.float64)
        ref, smax = att_reference(q[b].astype(np.float64), k, v, heads)
        check_rows(f"attention h{heads} hd{hd} Kk{kb} L{L}", got[b * L:(b + 1) * L, :A], ref,
                   RTOL_ATT * np.maximum(1.0, smax))


@pytest.mark.parametrize("heads", [1, 2, 3, 4])
@pytest.mark.parametrize("hd", [4, 8, 12, 16])
def test_attention(torch, seam, heads, hd):
    rng = np.random.default_rng(heads * 100 + hd)
    A = heads * hd
    for Kk, L in ((1, 65), (16, 64), (17, 130), (64, 200)):      # L = 64 and not a multiple of 64
        B = 2
        q = rng.standard_normal((B, L, A)).astype(np.float32)
        kv = rng.standard_normal((B, Kk, 2 * A)).astype(np.float32)
        run_attention(torch, seam, q, kv, heads, hd, Kk)


def test_attention_ragged_keys(torch, seam):
    """Each utterance attends to its own first K2 keys; the keys and values past them are NaN."""
    rng = np.random.default_rng(11)
    heads, hd, Kk, L = 4, 12, 64, 97
    Ks = [64, 16, 17, 1]
    B, A = len(Ks), heads * hd
    q = rng.standard_normal((B, L, A)).astype(np.float32)
    kv = np.full((B, Kk, 2 * A), np.nan, np.float32)
    for b, kb in enumerate(Ks):
        kv[b, :kb] = rng.standard_normal((kb, 2 * A))
    run_attention(torch, seam, q, kv, heads, hd, Kk, Ks=Ks)


def test_attention_large_scores(torch, seam):
    """Scores around 1e3: exp without the max shift overflows to inf."""
    rng = np.random.default_rng(12)
    heads, hd, Kk, L = 4, 16, 64, 70
    A = heads * hd
    q = (rng.standard_normal((1, L, A)) * 8.0).astype(np.float32)
    kv = (rng.standard_normal((1, Kk, 2 * A))).astype(np.float32)
    kv[..., :A] *= np.float32(32.0)
    run_attention(torch, seam, q, kv, heads, hd, Kk)


def test_attention_declines_past_48k_shared(torch, seam):
    q, o = torch.zeros(8, 64, device="cuda"), torch.zeros(8, 64, device="cuda")
    kv = torch.ones(97, 128, device="cuda")
    rc, _ = seam("attention", x=q, ldx=64, kv=kv, y=o, ldy=64, B=1, L=8, K=96, heads=4, hd=16)
    assert rc == OK and bool((o == 1).all())                 # 96 x 128 floats = 48 KB exactly
    rc, _ = seam("attention", x=q, ldx=64, kv=kv, y=o, ldy=64, B=1, L=8, K=97, heads=4, hd=16)
    assert rc == ERR_UNSUPPORTED


# ------------------------------------------------------------------ gate_mix ---------------------
@pytest.mark.parametrize("M,C", [(37, 100), (5, 64), (129, 192), (3, 7)])
def test_gate_mix(torch, seam, M, C):
    """C not a multiple of 64, M C not a multiple of 256, gate logits of +-80 (the gate saturates)."""
    rng = np.random.default_rng(M * C)
    f3 = rng.standard_normal((M, 3 * C)).astype(np.float32)
    f3[:, :C] *= np.float32(4.0)
    f3[::3, :C:2] = np.float32(80.0)
    f3[1::3, :C:3] = np.float32(-80.0)
    out = torch.full((M * C + 300,), SENT, device="cuda")
    rc, _ = seam("gate_mix", x=dev(torch, f3), y=out, M=M, C=C)
    assert rc == OK
    got = out.cpu().numpy()
    f = f3.astype(np.float64)
    s = O.sigmoid(f[:, :C])
    ref = s * f[:, C:2 * C] + (1.0 - s) * f[:, 2 * C:]
    check_rows(f"gate_mix M{M} C{C}", got[:M * C].reshape(M, C), ref, RTOL_MIX)
    assert (got[M * C:] == SENT).all()


# ------------------------------------------------------------------ greedy decode ----------------
def tie_logits(rng, M, V):
    """Random logits with exact ties of the row maximum placed across lanes and rounds of the warp's scan, and
    rows of -inf."""
    x = rng.standard_normal((M, V)).astype(np.float32)
    for m in range(M):
        if V > 1 and m % 3 == 0:
            k = min(V, 2 + m % 5)
            idx = rng.choice(V, size=k, replace=False)
            x[m, idx] = x[m].max() + np.float32(1.0)
        elif V > 33 and m % 3 == 1:                          # same lane, different rounds / different lanes
            j = int(rng.integers(0, V - 32))
            x[m, [j, j + 32 if m % 2 else j + 1]] = x[m].max() + np.float32(1.0)
    x[M // 2] = -np.inf
    return x


@pytest.mark.parametrize("V", [1, 31, 32, 33, 1000, 1024])
def test_argmax(torch, seam, V):
    rng = np.random.default_rng(V)
    M = 203
    x = tie_logits(rng, M, V)
    pred = torch.full((M + 5,), ISENT, dtype=torch.int32, device="cuda")
    rc, _ = seam("argmax", x=dev(torch, x), pred=pred, M=M, V=V)
    assert rc == OK
    got = pred.cpu().numpy()
    import torch as T
    assert np.array_equal(got[:M], T.argmax(T.from_numpy(x), dim=1).numpy())
    assert np.array_equal(got[:M], np.argmax(x, axis=1))
    assert (got[M:] == ISENT).all()


def amax_parts(x):
    """The CTC head's argmax partials: per slot p (columns 64 p .. 64 p + 63) the max and first argmax; -1 (with a
    value the merge must ignore) where the slot holds no column."""
    M, V = x.shape
    slots = 2 * ((V + 127) // 128)
    val = np.full((slots, M), np.float32(3e38))
    idx = np.full((slots, M), -1, np.int32)
    for p in range(slots):
        lo, hi = 64 * p, min(64 * p + 64, V)
        if lo < hi:
            val[p] = x[:, lo:hi].max(axis=1)
            idx[p] = lo + x[:, lo:hi].argmax(axis=1)
    return val, idx, slots


def decode_expect(pred, L, Lb, blank, collapse):
    toks = O.collapse_tokens(pred[:Lb], blank, bool(collapse))
    return toks + [-1] * (L - len(toks))


@pytest.mark.parametrize("L", [31, 32, 33, 1003])
@pytest.mark.parametrize("parts", [False, True])
@pytest.mark.parametrize("blank,collapse", [(0, 1), (5, 1), (5, 0)])
def test_ctc_collapse(torch, seam, L, parts, blank, collapse):
    """Greedy decode as the engine runs it: from an argmax (parts=False), or from the projection's per-slot
    partials (parts=True), with ragged lengths; compared with O.ctc_greedy_decode."""
    rng = np.random.default_rng(L * 7 + blank + 3 * collapse + int(parts))
    B, V = 3, 1030 if parts else 12
    Ls = [L, max(L - 17, 1), 1]
    # few distinct winners so that runs and repeats happen; ties between slots for the partials
    x = rng.standard_normal((B * L, V)).astype(np.float32)
    win = rng.integers(0, 8, size=B * L)
    win = np.where(rng.random(B * L) < 0.5, blank, win)
    x[np.arange(B * L), win] = 10.0
    ties = np.arange(0, B * L, 4)
    x[ties, (win[ties] + 64 * (1 + ties % 3)) % V] = 10.0   # the same maximum in a later slot
    pred_ref = np.argmax(x, axis=1).astype(np.int32)
    for b in range(B):
        full = O.ctc_greedy_decode(x[b * L:(b + 1) * L][None, :Ls[b]], blank, bool(collapse))[0]
        assert full == O.collapse_tokens(pred_ref[b * L:b * L + Ls[b]], blank, bool(collapse))
    rag = rag_dims(torch, B, RAG_L=Ls)
    tokens = torch.full((B * L + 5,), ISENT, dtype=torch.int32, device="cuda")
    lens = torch.full((B + 2,), ISENT, dtype=torch.int32, device="cuda")
    if parts:
        val, idx, slots = amax_parts(x)
        assert (idx == -1).any()
        pred = torch.full((B * L + 5,), ISENT, dtype=torch.int32, device="cuda")
        rc, _ = seam("ctc_collapse", pred=pred, tokens=tokens, lens=lens, B=B, L=L, blank=blank, collapse=collapse,
                     rag=rag, amax_val=dev(torch, val), amax_idx=dev(torch, idx), slots=slots)
    else:
        pred = dev(torch, np.concatenate([pred_ref, np.full(5, ISENT, np.int32)]))
        rc, _ = seam("ctc_collapse", pred=pred, tokens=tokens, lens=lens, B=B, L=L, blank=blank, collapse=collapse,
                     rag=rag)
    assert rc == OK
    p, t, n = pred.cpu().numpy(), tokens.cpu().numpy(), lens.cpu().numpy()
    for b in range(B):
        want = decode_expect(pred_ref[b * L:(b + 1) * L], L, Ls[b], blank, collapse)
        assert t[b * L:(b + 1) * L].tolist() == want, f"utterance {b}"
        assert n[b] == sum(1 for v in want if v >= 0)
        if parts:
            assert np.array_equal(p[b * L:b * L + Ls[b]], pred_ref[b * L:b * L + Ls[b]])
            assert (p[b * L + Ls[b]:(b + 1) * L] == ISENT).all()
    assert (t[B * L:] == ISENT).all() and (n[B:] == ISENT).all() and (p[B * L:] == ISENT).all()


@pytest.mark.parametrize("L", [1, 31, 32, 33, 1003])
@pytest.mark.parametrize("blank", [0, 5])
def test_ctc_runs(torch, seam, L, blank):
    """Timestamps: runs start and end at the utterance's first and last frame too."""
    rng = np.random.default_rng(L + blank)
    B, V = 3, 9
    x = rng.standard_normal((B, L, V)).astype(np.float32)
    win = rng.integers(0, V, size=(B, L))
    win = np.repeat(win, 3, axis=1)[:, :L]                   # runs of three
    win[:, 0] = (blank + 1) % V
    win[:, -1] = (blank + 2) % V
    win[1] = blank                                           # an utterance of blanks only
    win[2, :L // 2] = (blank + 3) % V                        # a run from the first frame
    x[np.arange(B)[:, None], np.arange(L)[None, :], win] = 10.0
    pred = dev(torch, np.argmax(x, axis=2).astype(np.int32).reshape(-1))
    mk = lambda: torch.full((B * L + 3,), ISENT, dtype=torch.int32, device="cuda")
    tokens, starts, ends = mk(), mk(), mk()
    lens = torch.full((B + 1,), ISENT, dtype=torch.int32, device="cuda")
    rc, _ = seam("ctc_runs", pred=pred, tokens=tokens, starts=starts, ends=ends, lens=lens, B=B, L=L, blank=blank)
    assert rc == OK
    t, s, e, n = (a.cpu().numpy() for a in (tokens, starts, ends, lens))
    for b, (toks, stamps) in enumerate(O.ctc_greedy_decode_with_timestamps(x, blank)):
        k = len(toks)
        assert n[b] == k
        row = slice(b * L, (b + 1) * L)
        assert t[row].tolist() == toks + [-1] * (L - k)
        assert s[row].tolist() == [a for a, _ in stamps] + [-1] * (L - k)
        assert e[row].tolist() == [z for _, z in stamps] + [-1] * (L - k)
    for a in (t, s, e):
        assert (a[B * L:] == ISENT).all()
    assert n[B] == ISENT


# ------------------------------------------------------------------ minmax / set_qparams ---------
@pytest.mark.parametrize("M,ld,c0,nc,const", [(37, 100, 13, 51, False), (1000, 192, 0, 192, False),
                                             (3, 20, 5, 7, True), (1, 8, 7, 1, False)])
def test_minmax_qparams(torch, seam, M, ld, c0, nc, const):
    """min / max over a column window of strided rows (+-1e30 outside it), then scale = max((max - min) / 255, 1e-10),
    zp = 0 - min / scale in fp32 (quantize.py:116-121), bit for bit."""
    rng = np.random.default_rng(M + nc)
    x = np.where(np.arange(M * ld).reshape(M, ld) % 2 == 0, np.float32(1e30), np.float32(-1e30)).astype(np.float32)
    x[:, c0:c0 + nc] = np.float32(2.5) if const else rng.standard_normal((M, nc)) * 3.0 + 1.0
    mm = torch.full((4,), SENT, device="cuda")
    qs = torch.full((ld + 2,), SENT, device="cuda")
    qz = torch.full((ld + 2,), SENT, device="cuda")
    rc, _ = seam("minmax", x=dev(torch, x), ldx=ld, M=M, c0=c0, nc=nc, mm=mm, q_scale=qs, q_zp=qz)
    assert rc == OK
    win = x[:, c0:c0 + nc]
    lo, hi = win.min(), win.max()
    f32 = np.float32
    scale = np.maximum((hi - lo) / f32(255.0), f32(1e-10)).astype(f32)
    zp = (f32(0.0) - lo / scale).astype(f32)
    got_mm, got_s, got_z = mm.cpu().numpy(), qs.cpu().numpy(), qz.cpu().numpy()
    assert got_mm[0] == lo and got_mm[1] == hi and (got_mm[2:] == SENT).all()
    if const:
        assert scale == f32(1e-10)
    assert (got_s[c0:c0 + nc] == scale).all() and (got_z[c0:c0 + nc] == zp).all()
    outside = np.r_[0:c0, c0 + nc:ld + 2]
    assert (got_s[outside] == SENT).all() and (got_z[outside] == SENT).all()


# ------------------------------------------------------------------ log-mel ----------------------
def mel_check(va, audio, n_mels):
    import torch as T
    from velocity_asr.audio import frontend_tables
    fb, win = frontend_tables(n_mels)
    got = va.compute_mel_spectrogram(T.from_numpy(audio).cuda(), n_mels=n_mels).cpu().numpy()
    raw = O.log_mel(audio.astype(np.float64), n_mels=n_mels, filters=fb.numpy(), window=win.numpy(), normalize=False)
    # O.log_mel's normalisation, except that a bin constant over time (an all-zero filter row, which n_mels >= 90
    # has, or digital silence) is exactly 0: fp64 rounding of its mean leaves up to 2e-4 / (std + 1e-10) otherwise
    d = raw - raw.mean(axis=1, keepdims=True)
    d[np.broadcast_to((raw == raw[:, :1]).all(axis=1, keepdims=True), d.shape)] = 0.0
    ref = d / (raw.std(axis=1, ddof=1, keepdims=True) + 1e-10)
    assert got.shape == ref.shape
    assert np.isfinite(got).all()
    err = float(np.abs(got - ref).max())
    log = os.environ.get("VASR_ERR_LOG")
    if log:
        with open(log, "a") as f:
            f.write(f"mel n{n_mels} S{audio.shape[-1]}\t{err:.3e}\t{err / MEL_ATOL:.3f}\n")
    assert err <= MEL_ATOL, f"n_mels {n_mels} S {audio.shape[-1]}: {err:.3e}"
    return got


@pytest.mark.parametrize("n_mels", [40, 64, 90, 100, 128])
def test_log_mel_widths(torch, n_mels):
    """The statistics merge runs G = 4, 4, 2, 2, 2 partial sums per bin for these widths, and the scalar
    normalisation path runs where n_mels % 4 != 0 (90).  Lengths: S in {201, 359, 360, 401} (two and three
    frames), and S with T % 32 in {0, 1, 31} (a last block of 32, 1 and 31 frames)."""
    import velocity_asr as va
    rng = np.random.default_rng(n_mels)
    for S in (201, 359, 360, 401, 4960, 5120, 4800, 16160):
        audio = (rng.standard_normal((2, S)) * 0.1).astype(np.float32)
        mel_check(va, audio, n_mels)


def test_log_mel_silence_and_scale(torch):
    """Digital silence inside an utterance gives exactly log(1e-10) before the normalisation; an all-zero utterance
    gives 0, not NaN; int16-scale amplitudes."""
    import torch as T
    import velocity_asr as va
    rng = np.random.default_rng(5)
    S = 16000
    audio = (rng.standard_normal((3, S)) * 0.1).astype(np.float32)
    audio[0, 4000:9000] = 0.0
    audio[1] = 0.0
    audio[2] *= np.float32(32768.0)
    for n_mels in (80, 90):
        got = mel_check(va, audio, n_mels)
        assert (got[1] == 0).all()
    raw = va.compute_mel_spectrogram(T.from_numpy(audio).cuda(), normalize=False).cpu().numpy()
    sil = raw[0, 4000 // 160 + 3:9000 // 160 - 2]               # frames whose 400 samples are all zero
    assert (sil == sil[0, 0]).all()
    assert abs(float(sil[0, 0]) - np.log(1e-10)) <= 2 * np.spacing(np.float32(23.0))   # logf(1e-10f), to an ulp


def test_log_mel_declines_129_bins(torch):
    import torch as T
    import velocity_asr as va
    with pytest.raises(NotImplementedError):
        va.compute_mel_spectrogram(T.zeros(1, 1000).cuda(), n_mels=129)
