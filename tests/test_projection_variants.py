"""The tensor-core projection kernel (csrc/gemm_tc.cu) one template instantiation at a time.

`launch_gemm_tc` picks one of 50 instantiations of `gemm_tc_kernel` / `gemm_tc2_kernel` from the shape and the
epilogue a projection asks for.  The model reaches most of them only through whole-model tests at a 1e-3 tolerance,
where a 3xTF32 split that lost one of its three products (about 1e-3) would hide.  Here every instantiation is run
through the debug seam `vasr_debug_gemm` (csrc/engine.cu), which takes every GemmArgs field plus an SM-count
override and reports the instantiation it launched, and each result is compared with an fp64 reference built from
the numpy oracle:
  * per row, error <= 5e-6 of the row's max |reference| (1e-5 with the folded LayerNorm), or of the row's max
    |pre-activation| where that is larger: the bar is the projection's, and every activation here has a slope of at
    most 1.13, so a sigmoid that squashes a 1e4-scaled row to 1 still carries the projection's absolute error (the
    gate's bar grows by 0.25 |l - t|, the mix's sensitivity to its logit);
  * FakeQuantize lands on the reference's grid point (one step allowed only where the reference value lies within
    rounding reach of a boundary; integer inputs with exact ties must round half to even);
  * NaN in every gap of A and of the residual, a sentinel around C: nothing outside the output is written and no
    output is NaN;
  * the bit-for-bit claims of DESIGN.md: a row's result does not depend on M (across the W-resident threshold too),
    on the grid size or on pair / single-CTA kernel, and the argmax partials agree with the output they replace.
The CPU tests pin the reference itself against the oracle's CTC head, gated fusion and temporal binding.
"""
import ctypes
import dataclasses
from ctypes import c_float, c_int32, c_int64, c_void_p
from typing import Optional

import numpy as np
import pytest

import velocity_oracle as O

NONE, GELU, SOFTPLUS, SIGMOID = 0, 1, 2, 3
ACT_NAMES = {NONE: "none", GELU: "gelu", SOFTPLUS: "softplus", SIGMOID: "sigmoid"}
ACT_FN = {NONE: lambda v: v, GELU: O.gelu, SOFTPLUS: O.softplus, SIGMOID: O.sigmoid}
LNA, AMAX, GATE = 1, 2, 4            # epilogue bits of gemm_tc2_kernel (EPI_LNA, EPI_AMAX, EPI_GATE)
RTOL, RTOL_LNA = 5e-6, 1e-5
SENTINEL = np.float32(-7777.25)


# ------------------------------------------------------------------ the variant table -----------
# (family, tn, act, pe, resid, quant, wres, epi): family 1 = gemm_tc_kernel (single CTA), 2 = gemm_tc2_kernel (CTA
# pair); the other fields are the template arguments.  One entry per instantiation a launch site of launch_gemm_tc
# can launch, read off its dispatch:
def _single():
    out = [(1, 128, a, pe, rs, 0, 0, 0) for a in (NONE, GELU, SOFTPLUS, SIGMOID) for pe, rs in
           ((1, 1), (1, 0), (0, 1), (0, 0))]                                   # VASR_TC_CASE, not pair: 16
    return out + [(1, 128, GELU, 1, 0, 1, 0, 0), (1, 128, NONE, 0, 0, 1, 0, 0)]  # quant, not pair: 2


def _pair128():
    out = [(2, 128, a, pe, rs, 0, 0, 0) for a in (NONE, GELU, SOFTPLUS, SIGMOID) for pe, rs in
           ((1, 1), (1, 0), (0, 1), (0, 0))]                                   # VASR_TC_CASE, pair: 16
    out += [(2, 128, NONE, 0, 0, 0, 1, 0), (2, 128, GELU, 0, 0, 0, 1, 0)]      # W resident: 2
    out += [(2, 128, GELU, 1, 0, 1, 0, 0), (2, 128, NONE, 0, 0, 1, 0, 0)]      # quant, pair: 2
    out += [(2, 128, NONE, 0, 0, 0, w, e) for w in (1, 0) for e in (LNA | AMAX, LNA, AMAX)]   # lna || amax: 6
    return out


def _pair192():
    return [(2, 192, NONE, 0, 0, 0, 0, GATE), (2, 192, GELU, 0, 0, 0, 0, LNA), (2, 192, SOFTPLUS, 0, 0, 0, 0, 0),
            (2, 192, GELU, 0, 0, 0, 0, 0), (2, 192, NONE, 0, 1, 0, 0, 0), (2, 192, NONE, 0, 0, 0, 0, 0)]   # t192: 6


VARIANTS = _single() + _pair128() + _pair192()


def vname(v):
    fam, tn, act, pe, rs, qu, wr, epi = v
    parts = ["single" if fam == 1 else f"pair{tn}", ACT_NAMES[act]]
    parts += [n for n, f in (("pe", pe), ("resid", rs), ("quant", qu), ("wres", wr)) if f]
    parts += [n for n, b in (("lna", LNA), ("amax", AMAX), ("gate", GATE)) if epi & b]
    return "-".join(parts)


# ------------------------------------------------------------------ cases -----------------------
@dataclasses.dataclass
class Case:
    expect: tuple
    M: int
    N: int                      # columns of the projection (3 C for the gate)
    K: int
    act: int = NONE
    act_from: int = 0
    view: str = "gap"           # "dense" (lda = K), "gap" (lda = K + 8, NaN between), "conv" (lda = 160, K = 240)
    rpb: int = 0                # rows per batch (0: plain matrix); batches are separated by a NaN gap
    pe: bool = False
    resid: bool = False
    quant: Optional[str] = None  # "rand": calibrated scale / zero point; "ties": integer data on exact ties
    ln_offset: Optional[float] = None   # folded LayerNorm; rows of A are offset + N(0, 1)
    amax: bool = False
    gate: bool = False
    pad_c: int = 8              # ldc = output width + pad_c (sentinel columns)
    num_sms: int = 0            # 0: the device's count; 1: the single-CTA kernel
    seed: int = 0

    @property
    def tm(self):
        return 128 if self.expect[0] == 1 else 256

    @property
    def tn(self):
        return self.expect[1]

    def id(self):
        s = f"{vname(self.expect)}-M{self.M}-N{self.N}-K{self.K}"
        if self.act_from:
            s += f"-from{self.act_from}"
        if self.rpb:
            s += f"-rpb{self.rpb}"
        if self.view != "gap":
            s += "-" + self.view
        if self.quant:
            s += "-" + self.quant
        if self.ln_offset is not None:
            s += f"-off{self.ln_offset:g}"
        if self.num_sms:
            s += f"-sms{self.num_sms}"
        return s


def _v(fam, tn, act, pe=0, rs=0, qu=0, wr=0, epi=0):
    return (fam, tn, act, pe, rs, qu, wr, epi)


def _cases():
    C = []
    acts = (NONE, GELU, SOFTPLUS, SIGMOID)
    for fam, sms in ((1, 1), (2, 0)):
        for a in acts:
            # plain: for the pair kernel, N must not tile into 192-column tiles (N % 192 in 1..127), except sigmoid
            C.append(Case(_v(fam, 128, a), 257, 400, 240, a, seed=1))
            C.append(Case(_v(fam, 128, a), 31, 60, 36, a, act_from=36 if a else 0, view="dense", seed=2))
            C.append(Case(_v(fam, 128, a, rs=1), 255, 1000, 160, a, resid=True, seed=3))
            C.append(Case(_v(fam, 128, a, rs=1), 129, 4 if fam == 1 else 448, 96, a, resid=True,
                          act_from=64 if fam == 2 and a else 0, seed=4))
            # pos-enc: the temporal-binding conv view (overlapping rows, lda = 160, K = 240) and one-row batches
            C.append(Case(_v(fam, 128, a, pe=1), 258, 192, 240, a, view="conv", rpb=129, pe=True, seed=5))
            C.append(Case(_v(fam, 128, a, pe=1), 5, 60, 36, a, rpb=1, pe=True, act_from=36 if a else 0, seed=6))
            C.append(Case(_v(fam, 128, a, pe=1, rs=1), 258, 400, 240, a, view="conv", rpb=129, pe=True,
                          resid=True, seed=7))
            C.append(Case(_v(fam, 128, a, pe=1, rs=1), 5, 132, 768, a, rpb=1, pe=True, resid=True, seed=8))
        # FakeQuantize: the plain projection, and the temporal-binding conv (GELU + pos-enc)
        C.append(Case(_v(fam, 128, NONE, qu=1), 257, 400, 240, quant="rand", seed=9))
        C.append(Case(_v(fam, 128, NONE, qu=1), 31, 60, 36, quant="ties", seed=10))
        C.append(Case(_v(fam, 128, GELU, pe=1, qu=1), 258, 192, 240, GELU, view="conv", rpb=129, pe=True,
                      quant="rand", seed=11))
        C.append(Case(_v(fam, 128, GELU, pe=1, qu=1), 5, 60, 36, GELU, rpb=1, pe=True, quant="ties", seed=12))
    for c in C:
        if c.expect[0] == 1:
            c.num_sms = 1
    C.append(Case(_v(1, 128, NONE), 1, 4, 4, num_sms=1, seed=13))
    C.append(Case(_v(2, 128, SIGMOID), 256, 4, 768, SIGMOID, seed=14))
    C.append(Case(_v(2, 128, GELU, pe=1), 3755, 192, 240, GELU, view="conv", rpb=751, pe=True, seed=15))
    C.append(Case(_v(2, 128, SOFTPLUS), 257, 448, 192, SOFTPLUS, act_from=64, seed=16))
    # W resident: one pair per n-tile keeps W in the stage ring (k-blocks nkb = 1, 2, 3 and 6 of the 6 stages)
    C.append(Case(_v(2, 128, NONE, wr=1), 1000, 60, 36, num_sms=2, seed=17))
    C.append(Case(_v(2, 128, NONE, wr=1), 12016, 1000, 192, seed=18))
    C.append(Case(_v(2, 128, GELU, wr=1), 1000, 60, 96, GELU, num_sms=2, seed=19))
    C.append(Case(_v(2, 128, GELU, wr=1), 2000, 400, 4, GELU, num_sms=16, seed=20))
    # folded LayerNorm and / or argmax partials (128-column tiles, W resident with K = 192 or K <= 96 for AMAX)
    C.append(Case(_v(2, 128, NONE, wr=1, epi=LNA), 1000, 60, 192, ln_offset=30.0, num_sms=2, seed=21))
    C.append(Case(_v(2, 128, NONE, wr=1, epi=LNA), 2000, 400, 192, ln_offset=300.0, num_sms=16, seed=22))
    C.append(Case(_v(2, 128, NONE, wr=1, epi=LNA | AMAX), 1000, 60, 192, ln_offset=0.0, amax=True, num_sms=2,
                  seed=23))
    C.append(Case(_v(2, 128, NONE, wr=1, epi=LNA | AMAX), 12016, 1000, 192, ln_offset=30.0, amax=True, seed=24))
    C.append(Case(_v(2, 128, NONE, wr=1, epi=AMAX), 1000, 60, 4, amax=True, num_sms=2, seed=25))
    C.append(Case(_v(2, 128, NONE, wr=1, epi=AMAX), 2000, 400, 96, amax=True, num_sms=16, seed=26))
    C.append(Case(_v(2, 128, NONE, epi=LNA), 257, 1000, 384, ln_offset=30.0, seed=27))
    C.append(Case(_v(2, 128, NONE, epi=LNA), 31, 132, 160, ln_offset=300.0, seed=28))
    C.append(Case(_v(2, 128, NONE, epi=LNA), 129, 448, 768, ln_offset=0.0, seed=29))
    C.append(Case(_v(2, 128, NONE, epi=LNA | AMAX), 257, 1000, 384, ln_offset=300.0, amax=True, seed=30))
    C.append(Case(_v(2, 128, NONE, epi=LNA | AMAX), 255, 60, 192, ln_offset=30.0, amax=True, seed=31))
    C.append(Case(_v(2, 128, NONE, epi=AMAX), 257, 1000, 240, amax=True, seed=32))
    C.append(Case(_v(2, 128, NONE, epi=AMAX), 31, 60, 36, amax=True, seed=33))
    C.append(Case(_v(2, 128, NONE, epi=AMAX), 129, 132, 4, amax=True, seed=34))
    # 192-column tiles: N = 192 a + (0 or >= 128)
    C.append(Case(_v(2, 192, NONE), 257, 320, 240, seed=35))
    C.append(Case(_v(2, 192, NONE), 31, 132, 36, seed=36))
    C.append(Case(_v(2, 192, NONE), 255, 576, 192, view="dense", seed=37))
    C.append(Case(_v(2, 192, NONE, rs=1), 257, 512, 96, resid=True, seed=38))
    C.append(Case(_v(2, 192, NONE, rs=1), 129, 192, 4, resid=True, seed=39))
    C.append(Case(_v(2, 192, SOFTPLUS), 257, 512, 240, SOFTPLUS, act_from=128, seed=40))
    C.append(Case(_v(2, 192, SOFTPLUS), 31, 320, 36, SOFTPLUS, act_from=36, seed=41))
    C.append(Case(_v(2, 192, GELU), 257, 320, 192, GELU, seed=42))
    C.append(Case(_v(2, 192, GELU), 129, 576, 160, GELU, seed=43))
    C.append(Case(_v(2, 192, GELU, epi=LNA), 257, 512, 192, GELU, ln_offset=30.0, seed=44))
    C.append(Case(_v(2, 192, GELU, epi=LNA), 129, 132, 384, GELU, ln_offset=300.0, seed=45))
    C.append(Case(_v(2, 192, GELU, epi=LNA), 31, 576, 160, GELU, ln_offset=0.0, seed=46))
    # gated fusion: C channels = 64, 192, 320 (N = 3 C, always whole 192-column tiles)
    C.append(Case(_v(2, 192, NONE, epi=GATE), 257, 192, 160, gate=True, seed=47))
    C.append(Case(_v(2, 192, NONE, epi=GATE), 129, 576, 384, gate=True, seed=48))
    C.append(Case(_v(2, 192, NONE, epi=GATE), 31, 960, 768, gate=True, seed=49))
    return C


CASES = _cases()


def test_variant_table_matches_the_dispatch_count():
    """18 single-CTA + 26 pair-128 + 6 pair-192 distinct instantiations, and no duplicates."""
    assert (len(_single()), len(_pair128()), len(_pair192())) == (18, 26, 6)
    assert len(set(VARIANTS)) == len(VARIANTS) == 50


def test_every_variant_has_two_shapes_and_a_ragged_one():
    """Each table entry is expected by >= 2 cases of different shapes, one of them with a partial last m-tile and
    a partial last n-tile (the gate excepted: it exists for whole 192-column tiles only)."""
    for v in VARIANTS:
        cs = [c for c in CASES if c.expect == v]
        assert len({(c.M, c.N, c.K, c.rpb) for c in cs}) >= 2, vname(v)
        rows = lambda c: c.rpb or c.M
        ragged = [c for c in cs if rows(c) % c.tm and (c.N % c.tn or c.gate)]
        assert ragged, vname(v)
    assert {c.expect for c in CASES} == set(VARIANTS)


# ------------------------------------------------------------------ inputs ----------------------
def make_a(rng, M, K, view, rpb, offset=None, special=True, integer=False):
    """Storage of A (NaN wherever no row reads) and the (M, K) fp64 rows the kernel sees."""
    rpb = rpb or M
    nb = M // rpb
    lda = {"dense": K, "gap": K + 8, "conv": 160}[view]
    if view == "conv":
        assert K == 240
    span = (rpb - 1) * lda + K
    bstride = span + 12 if nb > 1 else span
    bstride = (bstride + 3) // 4 * 4
    size = (nb - 1) * bstride + span + 4
    store = np.full(size, np.nan, np.float32)
    starts = (np.arange(nb)[:, None] * bstride + np.arange(rpb)[None, :] * lda).reshape(-1)
    idx = starts[:, None] + np.arange(K)[None, :]
    if integer:
        store[idx] = rng.integers(-3, 4, size=idx.shape).astype(np.float32)
    else:
        store[idx] = rng.standard_normal(idx.shape).astype(np.float32) + np.float32(offset or 0.0)
        if special and M >= 8:
            for r in range(3, M, 37):
                store[idx[r]] *= np.float32(1e4)
            for r in range(7, M, 41):
                store[idx[r]] = 0.0
    return store, idx, lda, (bstride if nb > 1 else 0), store[idx].astype(np.float64)


def gate_weights(rng, C, K):
    """The unpermuted stacked fusion weight [gate (C x K) | local | global] and its bias."""
    w = (rng.standard_normal((3 * C, K)) / np.sqrt(K)).astype(np.float32)
    return w, rng.standard_normal(3 * C).astype(np.float32)


# ------------------------------------------------------------------ fp64 reference --------------
def fq_level_value(q, scale, zp):
    """The value of FakeQuantize level q as the fp32 operations (q - zp) * scale give it."""
    return ((q.astype(np.float32) - zp) * scale).astype(np.float64)


def fq_round(y, scale, zp):
    """FakeQuantize (asymmetric uint8, round half to even) of the fp64 value y: integer level and its value."""
    q = np.clip(np.rint(y / scale.astype(np.float64) + zp.astype(np.float64)), 0, 255)
    return q, fq_level_value(q, scale, zp)


def reference(A, W, b, *, act=NONE, act_from=0, quant=None, pe=None, resid=None, ln=None, gate=False, rpb=0):
    """fp64 epilogue(A W^T) in the order kernels.cuh documents: bias -> FakeQuantize -> activation on n >= act_from
    -> pos-enc -> residual; ln = (gamma, beta, eps): Linear(LayerNorm(A)); gate: sigmoid(g) l + (1 - sigmoid(g)) t
    over the three column thirds.  quant = (scale, zp, levels): levels (M, N) overrides the rounding."""
    with np.errstate(over="ignore"):       # sigmoid of the 1e4-scaled rows
        return _reference(A, W, b, act, act_from, quant, pe, resid, ln, gate, rpb)


def _reference(A, W, b, act, act_from, quant, pe, resid, ln, gate, rpb):
    W = W.astype(np.float64)
    b = None if b is None else b.astype(np.float64)
    x = O.layer_norm(A, ln[0].astype(np.float64), ln[1].astype(np.float64), ln[2]) if ln is not None else A
    y = O.linear(x, W, b)
    if quant is not None:
        scale, zp, q = quant
        if q is None:
            q, _ = fq_round(y, scale, zp)
        y = fq_level_value(q, scale, zp)
    if act != NONE:
        y = y.copy()
        y[:, act_from:] = ACT_FN[act](y[:, act_from:])
    if pe is not None:
        pe_time, pe_freq = pe
        half = pe_time.shape[1]
        rows = np.arange(A.shape[0]) % (rpb or A.shape[0])
        y = y + np.concatenate([pe_time[rows].astype(np.float64),
                                np.broadcast_to(pe_freq.astype(np.float64), (A.shape[0], pe_freq.size))], axis=1)
        assert half + pe_freq.size == y.shape[1]
    if resid is not None:
        y = y + resid
    if gate:
        C = y.shape[1] // 3
        s = O.sigmoid(y[:, :C])
        y = s * y[:, C:2 * C] + (1.0 - s) * y[:, 2 * C:]
    return y


def amax_reference(y, N):
    """Per row and slot p (columns 64 p .. 64 p + 63 of the output): (max, first argmax); -inf / -1 when empty."""
    slots = 2 * ((N + 127) // 128)
    val = np.full((slots, y.shape[0]), -np.inf)
    idx = np.full((slots, y.shape[0]), -1, np.int64)
    for p in range(slots):
        lo, hi = 64 * p, min(64 * p + 64, N)
        if lo < hi:
            val[p] = y[:, lo:hi].max(axis=1)
            idx[p] = lo + y[:, lo:hi].argmax(axis=1)
    return val, idx


# ------------------------------------------------------------------ reference pinned on the oracle (CPU)
@pytest.fixture(scope="module")
def model_sd():
    import torch
    import velocity_asr as va
    torch.manual_seed(0)
    m = va.VELOCITYASR(va.VelocityASRConfig())
    sd = {k: v.detach().numpy().astype(np.float64) for k, v in m.state_dict().items()}
    rng = np.random.default_rng(5)      # non-trivial LayerNorm parameters (init is gamma = 1, beta = 0)
    for k in sd:
        if ".norm" in k or "proj.0." in k:
            if k.endswith(".weight") and sd[k].ndim == 1:
                sd[k] = 1.0 + 0.3 * rng.standard_normal(sd[k].shape)
            elif k.endswith(".bias") and sd[k].ndim == 1:
                sd[k] = 0.3 * rng.standard_normal(sd[k].shape)
    return sd


def test_reference_matches_oracle_ctc_head(model_sd):
    sd = model_sd
    x = np.random.default_rng(1).standard_normal((2, 37, 192)) + 30.0
    ref = reference(x.reshape(-1, 192), sd["ctc_head.proj.2.weight"], sd["ctc_head.proj.2.bias"],
                    ln=(sd["ctc_head.proj.0.weight"], sd["ctc_head.proj.0.bias"], 1e-5))
    want = O.ctc_head(x, sd).reshape(-1, 1000)
    assert np.abs(ref - want).max() <= 1e-12 * np.abs(want).max()
    val, idx = amax_reference(ref, 1000)
    assert val.shape == (16, 74)
    best = np.argmax(val, axis=0)                                   # the best slot, ties to the lower one
    assert (idx[best, np.arange(74)] == want.argmax(axis=1)).all()


def test_reference_matches_oracle_gated_fusion(model_sd):
    sd, p, d = model_sd, "global_context.fusion.", 192
    rng = np.random.default_rng(2)
    loc, ctx = rng.standard_normal((1, 41, d)), rng.standard_normal((1, 41, d))
    # the stacked [gate | local | global] projection of [loc | ctx] the engine builds before permuting it
    w = np.zeros((3 * d, 2 * d))
    w[:d] = sd[p + "gate_proj.0.weight"]
    w[d:2 * d, :d] = sd[p + "local_proj.weight"]
    w[2 * d:, d:] = sd[p + "global_proj.weight"]
    b = np.concatenate([sd[p + "gate_proj.0.bias"], sd[p + "local_proj.bias"], sd[p + "global_proj.bias"]])
    mix = reference(np.concatenate([loc, ctx], -1)[0], w, b, gate=True)
    got = O.linear(mix, sd[p + "out_proj.weight"], sd[p + "out_proj.bias"])
    want = O.gated_fusion(loc, ctx, sd, p)[0]
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_reference_matches_oracle_temporal_binding(model_sd):
    """The conv as a projection over the overlapping view (lda = 160, K = 240) + GELU + pos-enc, then the LayerNorm."""
    sd, pfx = model_sd, "temporal_binding."
    rng = np.random.default_rng(3)
    B, T = 3, 51
    mel = rng.standard_normal((B, T, 80))
    L = (T - 1) // 2 + 1
    Tp = T + 2 + (T + 2) % 2
    pad = np.zeros((B, Tp, 80))
    pad[:, 1:T + 1] = mel
    flat = pad.reshape(-1)
    starts = (np.arange(B)[:, None] * Tp * 80 + np.arange(L)[None, :] * 160).reshape(-1)
    A = flat[starts[:, None] + np.arange(240)[None, :]]
    w = sd[pfx + "conv.weight"]                                          # (192, 80, 3)
    W = w.transpose(0, 2, 1).reshape(192, 240)                          # k = 80 j + c
    pe_time = sd[pfx + "pos_encoding.pe_time"][:L]
    pe_freq = sd[pfx + "pos_encoding.pe_freq"].reshape(-1)
    y = reference(A, W, sd[pfx + "conv.bias"], act=GELU, pe=(pe_time, pe_freq), rpb=L)
    got = O.layer_norm(y, sd[pfx + "norm.weight"], sd[pfx + "norm.bias"]).reshape(B, L, 192)
    want = O.temporal_binding(mel, sd)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_reference_fake_quantize_rounds_half_to_even():
    scale, zp = np.full(4, 0.5, np.float32), np.full(4, 128.5, np.float32)
    y = np.array([[0.0, 1.0, -1.0, 2.0]])                      # y / 0.5 + 128.5 = 128.5, 130.5, 126.5, 132.5
    q, dq = fq_round(y, scale, zp)
    assert q.tolist() == [[128, 130, 126, 132]]
    assert dq.tolist() == [[-0.25, 0.75, -1.25, 1.75]]
    assert (O.fake_quantize(y, scale.astype(np.float64), zp.astype(np.float64), symmetric=False) == dq).all()


# ------------------------------------------------------------------ the seam (GPU) --------------
class _GemmCall(ctypes.Structure):
    _fields_ = [("A", c_void_p), ("lda", c_int64), ("rows_per_batch", c_int64), ("batch_stride", c_int64),
                ("M", c_int64), ("N", c_int64), ("K", c_int64), ("C", c_void_p), ("ldc", c_int64),
                ("resid", c_void_p), ("ldr", c_int64), ("q_scale", c_void_p), ("q_zp", c_void_p),
                ("pe_time", c_void_p), ("pe_freq", c_void_p), ("pe_half", c_int64), ("pe_rows", c_int64),
                ("amax_val", c_void_p), ("amax_idx", c_void_p),
                ("W", c_void_p), ("bias", c_void_p), ("ln_gamma", c_void_p), ("ln_beta", c_void_p),
                ("ln_eps", c_float), ("act", c_int32), ("act_from", c_int32), ("gate", c_int32),
                ("num_sms", c_int32), ("stream", c_void_p), ("variant", c_int32 * 8)]


@pytest.fixture(scope="module")
def seam():
    import torch
    from velocity_asr import _native
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    fn = _native.lib().vasr_debug_gemm
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.POINTER(_GemmCall)]
    return fn


class Problem:
    """Inputs of one case on the host and the device, the call into the seam and the fp64 reference."""

    def __init__(self, c: Case):
        import torch
        rng = np.random.default_rng(1000 + c.seed)
        self.c = c
        integer = c.quant == "ties"
        self.store, self.idx, self.lda, self.bstride, self.A = make_a(
            rng, c.M, c.K, c.view, c.rpb, offset=c.ln_offset, integer=integer)
        if c.gate:
            self.W, self.b = gate_weights(rng, c.N // 3, c.K)
        elif integer:
            self.W = rng.integers(-2, 3, size=(c.N, c.K)).astype(np.float32)
            self.b = rng.integers(-4, 5, size=c.N).astype(np.float32)
        else:
            self.W = (rng.standard_normal((c.N, c.K)) / np.sqrt(c.K)).astype(np.float32)
            self.b = rng.standard_normal(c.N).astype(np.float32)
        self.ln = None
        if c.ln_offset is not None:
            self.ln = ((1.0 + 0.3 * rng.standard_normal(c.K)).astype(np.float32),
                       (0.3 * rng.standard_normal(c.K)).astype(np.float32), 1e-5)
        self.out_w = c.N // 3 if c.gate else c.N
        self.ldc = self.out_w + c.pad_c
        self.resid = self.ldr = None
        if c.resid:
            self.ldr = c.N + 12
            r = np.full((c.M, self.ldr), np.nan, np.float32)
            r[:, :c.N] = rng.standard_normal((c.M, c.N))
            self.resid = r
        self.pe = None
        if c.pe:
            rows = c.rpb or c.M
            half = (c.N // 2 + 3) // 4 * 4
            self.pe = (O.positional_time_table(rows, 2 * half, dtype=np.float32),
                       rng.standard_normal(c.N - half).astype(np.float32))
        self.quant = None
        if c.quant == "rand":
            pre = reference(self.A, self.W, self.b)
            normal = np.abs(self.A).max(axis=1) < 100       # scale from the N(0, 1) rows: the 1e4 rows clamp
            lo, hi = pre[normal].min(axis=0), pre[normal].max(axis=0)
            scale = np.maximum((hi - lo) / 255, 1e-10).astype(np.float32)
            self.quant = (scale, (0 - lo / scale).astype(np.float32))
        elif c.quant == "ties":
            # integer pre-activations y: y / 0.5 + zp is a tie (k + 0.5) for every y; half to even decides
            self.quant = (np.full(c.N, 0.5, np.float32), np.full(c.N, 128.5, np.float32))
        dev = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.d_store = dev(self.store)
        self.d_resid = dev(self.resid)
        self.d_pe = (dev(self.pe[0]), dev(self.pe[1])) if self.pe else (None, None)
        self.d_q = (dev(self.quant[0]), dev(self.quant[1])) if self.quant else (None, None)

    def run(self, seam, num_sms=None, M=None, amax=None):
        """One call; returns (status, variant, C buffer, amax_val, amax_idx).  M < c.M: the first M rows only."""
        import torch
        c = self.c
        M = c.M if M is None else M
        amax = c.amax if amax is None else amax
        rpb = c.rpb
        assert M % (rpb or 1) == 0
        C = torch.full((M + 3, self.ldc), float(SENTINEL), device="cuda")
        slots = 2 * ((c.N + 127) // 128)
        av = torch.full((slots * M + 64,), float(SENTINEL), device="cuda") if amax else None
        ai = torch.full((slots * M + 64,), -7, dtype=torch.int32, device="cuda") if amax else None
        W = np.ascontiguousarray(self.W)
        b = np.ascontiguousarray(self.b)
        g = _GemmCall()
        g.A = self.d_store.data_ptr(); g.lda = self.lda; g.rows_per_batch = rpb
        g.batch_stride = self.bstride if rpb else 0
        g.M, g.N, g.K = M, c.N, c.K
        g.C = C.data_ptr(); g.ldc = self.ldc
        if self.d_resid is not None:
            g.resid = self.d_resid.data_ptr(); g.ldr = self.ldr
        if self.quant:
            g.q_scale, g.q_zp = self.d_q[0].data_ptr(), self.d_q[1].data_ptr()
        if self.pe:
            g.pe_time, g.pe_freq = self.d_pe[0].data_ptr(), self.d_pe[1].data_ptr()
            g.pe_half, g.pe_rows = self.pe[0].shape[1], rpb or M
        if amax:
            g.amax_val, g.amax_idx = av.data_ptr(), ai.data_ptr()
        g.W = W.ctypes.data; g.bias = b.ctypes.data
        if self.ln is not None:
            gam, bet = np.ascontiguousarray(self.ln[0]), np.ascontiguousarray(self.ln[1])
            g.ln_gamma, g.ln_beta, g.ln_eps = gam.ctypes.data, bet.ctypes.data, self.ln[2]
        g.act, g.act_from, g.gate = c.act, c.act_from, int(c.gate)
        g.num_sms = c.num_sms if num_sms is None else num_sms
        g.stream = torch.cuda.current_stream().cuda_stream
        rc = seam(ctypes.byref(g))
        torch.cuda.synchronize()
        return rc, tuple(g.variant), C.cpu().numpy(), (None if av is None else av.cpu().numpy()), \
            (None if ai is None else ai.cpu().numpy())

    def pre(self):
        """The projection before FakeQuantize, activation, pos-enc, residual and gate mix."""
        return reference(self.A, self.W, self.b, ln=self.ln)

    def ref(self, M=None, q_levels=None):
        c = self.c
        M = c.M if M is None else M
        rpb = c.rpb or M
        quant = (self.quant[0], self.quant[1], q_levels) if self.quant else None
        return reference(self.A[:M], self.W, self.b, act=c.act, act_from=c.act_from, quant=quant,
                         pe=self.pe, resid=None if self.resid is None else self.resid[:M, :c.N].astype(np.float64),
                         ln=self.ln, gate=c.gate, rpb=rpb)


def row_scale(ref, pre):
    """Per row: the larger of max |output| and max |pre-activation| (see the module docstring)."""
    return np.maximum(np.abs(ref).max(axis=1, keepdims=True), np.abs(pre).max(axis=1, keepdims=True))


def assert_rows_close(out, ref, rtol, what, scale):
    assert not np.isnan(out).any(), f"{what}: NaN in the output"
    err = np.abs(out.astype(np.float64) - ref)
    lim = np.broadcast_to(rtol * scale, err.shape)
    bad = np.argwhere(err > lim)
    if bad.size:
        r, n = bad[0]
        raise AssertionError(f"{what}: {len(bad)} elements off, first at row {r} col {n}: got {out[r, n]!r}, "
                             f"fp64 {ref[r, n]!r}, error {err[r, n] / max(lim[r, n] / rtol, 1e-300):.3g} of the "
                             f"row scale (bar {rtol:g})")


def check_sentinels(Cbuf, M, width, what):
    assert (Cbuf[:M, width:] == SENTINEL).all(), f"{what}: wrote past column {width} (ldc padding)"
    assert (Cbuf[M:] == SENTINEL).all(), f"{what}: wrote past row {M}"


def check_case(p: Problem, Cbuf, av, ai, what):
    c = p.c
    M, N = c.M, c.N
    rtol = RTOL_LNA if c.ln_offset is not None else RTOL
    if c.amax:
        assert (Cbuf == SENTINEL).all(), f"{what}: the argmax epilogue wrote the output"
        slots = 2 * ((N + 127) // 128)
        val, idx = av[:slots * M].reshape(slots, M), ai[:slots * M].reshape(slots, M)
        assert (av[slots * M:] == SENTINEL).all() and (ai[slots * M:] == -7).all(), f"{what}: wrote past the slots"
        ref = p.ref()
        rv, ri = amax_reference(ref, N)
        empty = ri < 0
        assert (idx[empty] == -1).all() and np.isneginf(val[empty]).all(), f"{what}: empty slot not (-inf, -1)"
        lim = rtol * np.abs(ref).max(axis=1)[None, :]
        assert (np.abs(val[~empty] - rv[~empty]) <= np.broadcast_to(lim, val.shape)[~empty]).all(), f"{what}: slot max"
        # the index names a column of the slot whose reference value is a maximum within the tolerance
        slot_of = np.where(empty, -1, idx // 64)
        assert (slot_of == np.where(empty, -1, np.arange(slots)[:, None])).all(), f"{what}: index outside its slot"
        picked = ref[np.arange(M)[None, :].repeat(slots, 0)[~empty], idx[~empty]]
        assert (np.abs(picked - rv[~empty]) <= 2 * np.broadcast_to(lim, val.shape)[~empty]).all(), \
            f"{what}: argmax column is not a maximum"
        return
    out = Cbuf[:M, :p.out_w]
    check_sentinels(Cbuf, M, p.out_w, what)
    if not c.quant:
        ref, pre = p.ref(), p.pre()
        scale = row_scale(ref, pre)
        if c.gate:
            # an error dg of the gate logit moves s l + (1 - s) t by up to 0.25 |l - t| dg
            C3 = c.N // 3
            scale = scale * (1.0 + 0.25 * np.abs(pre[:, C3:2 * C3] - pre[:, 2 * C3:]))
        assert_rows_close(out, ref, rtol, what, scale)
        return
    # FakeQuantize: the pre-activation levels of the kernel must be the reference's, except that a value whose fp64
    # reference lies within rounding reach of a level boundary may take the neighbouring level.  Rounding reach is
    # 1e-5 of a step, or the kernel's own fp32-grade error on the value (the 5e-6 bar) if larger; with integer data
    # (exact ties) the pre-activation is exact and no neighbour is allowed.
    scale, zp = p.quant
    pre = reference(p.A, p.W, p.b)
    t = pre / scale.astype(np.float64) + zp.astype(np.float64)
    q0 = np.clip(np.rint(t), 0, 255)
    if c.quant == "ties":
        near = np.zeros_like(t, bool)
    else:
        reach = np.maximum(1e-5, RTOL * np.abs(pre).max(axis=1, keepdims=True) / scale.astype(np.float64))
        near = np.abs(np.abs(t - np.floor(t)) - 0.5) < reach
    cands = [q0] + [np.clip(q0 + d, 0, 255) for d in (-1, 1)]
    refs = [p.ref(q_levels=q) for q in cands]
    if c.act == NONE and not c.pe:
        # the grid point itself: x + (dq - x) in fp32 leaves at most two roundings of max(|x|, |dq|)
        tols = [2.0 ** -21 * np.maximum(np.abs(pre), np.abs(r)) for r in refs]
        if c.quant == "ties":
            tols = [np.zeros_like(pre)] * 3
    else:
        # the activation (slope <= 1.13) also carries the rounding of x + (dq - x)
        dqs = [fq_level_value(q, scale, zp) for q in cands]
        tols = [RTOL * row_scale(r, pre) + 1.13 * 2.0 ** -21 * np.maximum(np.abs(pre), np.abs(d))
                for r, d in zip(refs, dqs)]
    o = out.astype(np.float64)
    assert not np.isnan(out).any(), f"{what}: NaN in the output"
    ok = np.abs(o - refs[0]) <= tols[0]
    for r, tl in zip(refs[1:], tols[1:]):
        ok |= near & (np.abs(o - r) <= tl)
    bad = np.argwhere(~ok)
    if bad.size:
        r, n = bad[0]
        raise AssertionError(f"{what}: {len(bad)} FakeQuantize outputs off the grid, first at row {r} col {n}: got "
                             f"{out[r, n]!r}, level {q0[r, n]:g} -> {refs[0][r, n]!r} (x / scale + zp = {t[r, n]!r})")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id() for c in CASES])
def test_projection_variant(seam, case):
    p = Problem(case)
    rc, variant, Cbuf, av, ai = p.run(seam)
    assert rc == 0, f"vasr_debug_gemm returned {rc}"
    assert variant in VARIANTS, f"launched {variant}, which is not in the variant table"
    assert variant == case.expect, f"launched {vname(variant)}, expected {vname(case.expect)}"
    check_case(p, Cbuf, av, ai, case.id())


# ------------------------------------------------------------------ bit-for-bit invariants -------
def _find(expect, **kw):
    for c in CASES:
        if c.expect == expect and all(getattr(c, k) == v for k, v in kw.items()):
            return c
    raise LookupError(expect)


# (a) the rows of a projection give the same bits whatever M is (the row count crosses the W-resident threshold in
# the first two: 12016 rows take one pair per n-tile with W resident, 257 rows the round-robin walk)
ROW_CASES = [
    _find(_v(2, 128, NONE, wr=1), M=12016),
    _find(_v(2, 128, NONE, wr=1, epi=LNA | AMAX), M=12016),
    _find(_v(2, 192, GELU, epi=LNA), M=257),
    _find(_v(2, 192, NONE, epi=GATE), M=257),
    _find(_v(2, 128, SIGMOID, pe=1, rs=1), M=258),
    _find(_v(1, 128, SOFTPLUS, rs=1), M=255),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ROW_CASES, ids=[c.id() for c in ROW_CASES])
def test_rows_do_not_depend_on_m(seam, case):
    p = Problem(case)
    rc, v_full, full, _, _ = p.run(seam, amax=False)
    assert rc == 0
    step = case.rpb or 1
    for M in (1, 129, 257):
        M = max(step, M // step * step)
        if M >= case.M:
            continue
        rc, v, part, _, _ = p.run(seam, M=M, amax=False)
        assert rc == 0
        w = p.out_w
        assert np.array_equal(part[:M, :w].view(np.uint32), full[:M, :w].view(np.uint32)), \
            f"rows 0..{M} differ between M = {M} ({vname(v)}) and M = {case.M} ({vname(v_full)})"


# (b) the grid size does not change a bit: the device's SM count, 16 and 2 (pair kernel; a small grid walks many
# tiles per pair) and 1 (the single-CTA kernel, which declines the LayerNorm, argmax and gate epilogues)
SMS_CASES = [
    _find(_v(2, 128, NONE, wr=1), M=12016),
    _find(_v(2, 128, GELU, wr=1), M=2000),
    _find(_v(2, 128, SOFTPLUS, rs=1), M=255),
    _find(_v(2, 128, GELU, pe=1, qu=1), M=258),
    _find(_v(2, 192, NONE), M=257),
    _find(_v(2, 192, SOFTPLUS), M=257),
    _find(_v(2, 192, GELU), M=129),
    _find(_v(2, 192, NONE, rs=1), M=257),
    _find(_v(2, 128, NONE, epi=LNA), M=257),
    _find(_v(2, 192, GELU, epi=LNA), M=257),
    _find(_v(2, 192, NONE, epi=GATE), M=257),
    _find(_v(2, 128, NONE, wr=1, epi=LNA | AMAX), M=1000),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", SMS_CASES, ids=[c.id() for c in SMS_CASES])
def test_grid_size_does_not_change_bits(seam, case):
    p = Problem(case)
    fused = case.ln_offset is not None or case.amax or case.gate
    runs = {}
    for sms in (0, 16, 2, 1):
        rc, v, Cbuf, av, ai = p.run(seam, num_sms=sms)
        if sms == 1 and fused:
            assert rc == 5 and v == (0,) * 8, "the single-CTA kernel has no fused LayerNorm / argmax / gate"
            continue
        assert rc == 0 and v in VARIANTS, (sms, v)
        assert (v[0] == 1) == (sms == 1)
        check_case(p, Cbuf, av, ai, f"{case.id()} sms={sms}")
        runs[sms] = (v, Cbuf, av, ai)
    v0, C0, av0, ai0 = runs[0]
    for sms, (v, Cb, av, ai) in runs.items():
        same = np.array_equal(Cb.view(np.uint32), C0.view(np.uint32))
        if av0 is not None:
            same = same and np.array_equal(av.view(np.uint32), av0.view(np.uint32)) and np.array_equal(ai, ai0)
        assert same, f"num_sms {sms} ({vname(v)}) and the device count ({vname(v0)}) give different bits"


# (c) the argmax partials against the output they stand for: the same inputs without the argmax epilogue
AMAX_CASES = [c for c in CASES if c.amax]


def _check_partials(out, val, idx, N, what):
    M = out.shape[0]
    slots = 2 * ((N + 127) // 128)
    val, idx = val[:slots * M].reshape(slots, M), idx[:slots * M].reshape(slots, M)
    for p_ in range(slots):
        lo, hi = 64 * p_, min(64 * p_ + 64, N)
        if lo >= hi:
            assert (idx[p_] == -1).all() and np.isneginf(val[p_]).all(), f"{what}: slot {p_}"
            continue
        seg = out[:, lo:hi]
        mx = seg.max(axis=1)
        assert np.array_equal(val[p_].view(np.uint32), mx.view(np.uint32)), f"{what}: slot {p_} max is not the output's"
        assert (idx[p_] == lo + seg.argmax(axis=1)).all(), f"{what}: slot {p_} index is not the first maximum"
    # what the collapse kernel makes of them: the best slot, ties to the lower one
    best = np.zeros(M, np.int64)
    for p_ in range(1, slots):
        best = np.where(val[p_] > val[best, np.arange(M)], p_, best)
    assert (idx[best, np.arange(M)] == out[:, :N].argmax(axis=1)).all(), f"{what}: collapsed argmax"


@pytest.mark.gpu
@pytest.mark.parametrize("case", AMAX_CASES, ids=[c.id() for c in AMAX_CASES])
def test_argmax_partials_equal_the_output(seam, case):
    p = Problem(case)
    rc, v, _, av, ai = p.run(seam)
    assert rc == 0
    rc, v2, Cbuf, _, _ = p.run(seam, amax=False)
    assert rc == 0 and not (v2[7] & AMAX)
    _check_partials(Cbuf[:case.M, :case.N], av, ai, case.N, f"{vname(v)} vs {vname(v2)}")


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [(30, 31, 32, 33), (61, 62, 63, 64, 65), (125, 126, 127, 128, 129)],
                         ids=["chunk", "half", "ntile"])
@pytest.mark.parametrize("lna", [False, True], ids=["plain", "lna"])
def test_argmax_partials_exact_ties(seam, cols, lna):
    """Columns with zero weight rows and equal bias are exactly equal in every row and hold its maximum: ties across
    a 32-column chunk, the two halves of an n-tile, and two n-tiles."""
    case = Case(_v(2, 128, NONE, epi=(LNA | AMAX) if lna else AMAX), 257, 400, 192 if lna else 96, amax=True,
                ln_offset=30.0 if lna else None, seed=60)
    p = Problem(case)
    p.W[list(cols)] = 0.0
    p.b[list(cols)] = 50.0 if not lna else 0.0
    if lna:
        # b' = b + W beta = 0 on the tie columns; make them the maximum through the other columns instead
        p.b[:] = -50.0
        p.b[list(cols)] = 0.0
    rc, v, _, av, ai = p.run(seam)
    assert rc == 0 and v == case.expect
    rc, _, Cbuf, _, _ = p.run(seam, amax=False)
    assert rc == 0
    out = Cbuf[:case.M, :case.N]
    normal = np.abs(p.A).max(axis=1) < 100
    assert (out[normal][:, cols[0]] == out[normal][:, list(cols)].max(axis=1)).all()
    assert (out[normal].argmax(axis=1) == cols[0]).all(), "the tie columns are not the rows' maximum"
    _check_partials(out, av, ai, case.N, f"ties {cols}")


# declines: what launch_gemm_tc does not take comes back as VASR_ERR_UNSUPPORTED, not as a different kernel
DECLINES = [
    Case(_v(2, 128, NONE, epi=LNA), 129, 400, 128, ln_offset=0.0),           # K / 32 = 4 k-blocks: not > 4 A slots
    Case(_v(2, 128, GELU, epi=LNA), 129, 400, 192, GELU, ln_offset=0.0),     # LNA + GELU needs 192-column tiles
    Case(_v(2, 192, NONE, epi=GATE), 129, 480, 160, gate=True),              # 3 C = 480: not whole 192-column tiles
    Case(_v(2, 128, GELU, epi=AMAX), 129, 400, 96, GELU, amax=True),         # argmax of an activated output
    Case(_v(2, 128, GELU, rs=1, qu=1), 129, 400, 96, GELU, resid=True, quant="rand"),   # quant with residual
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", DECLINES, ids=[c.id() for c in DECLINES])
def test_unsupported_combinations_are_declined(seam, case):
    p = Problem(case)
    rc, v, Cbuf, av, ai = p.run(seam)
    assert rc == 5 and v == (0,) * 8, (rc, v)
    assert (Cbuf == SENTINEL).all()
