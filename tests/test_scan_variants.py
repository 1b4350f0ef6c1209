"""The selective scan (csrc/scan.cu) one kernel instantiation at a time, against fp64 references.

`launch_selective_scan` picks one of 18 kernels from the problem: `scan_rp_kernel` (structured A, N = 64, the
model's true recurrence) with one or two row pairs per lane, each unsplit or cut in time into slots that hand the
state over through global memory; `scan_seq_kernel` (generic A, N = 32 / 16, or rows the row-packed kernel cannot
take) in five CTA shapes, structured or generic; `scan_quirk_kernel` (the reference's default 'parallel' scan) for
N = 64 / 32 / 16, structured or generic.  The debug seam `vasr_debug_scan` (csrc/engine.cu) takes every ScanArgs
field, lets a test choose the row-packed shape and the split, and the SM count the split rule plans for, and reports
the instantiation it launched with its slot count.

What each comparison asserts:
  * per element, |got - ref| <= kappa * m, where m is the magnitude of the terms the output sums: for the true
    recurrence m[t] = sum_n habs[t, n] |C[t, n]| + |x D| with habs = exp(dt A) habs + |u B| carried next to h, for the
    quirk the same over the terms its rule adds (hP's terms q (H - pd H[parent]) with |H| and |pd H[parent]| counted
    apart, times 1 + |A| S for the fp32 rounding of the decay exponent), times |silu(z)| when gated; the quirk may
    also drop whole the terms whose decay exp(A S) is below 2^-126, which ex2.approx.ftz flushes to zero (its phases
    2 and 3 rest on that, and a switch while a term is still above it fails the bar).  The structured
    kernels carry the state divided by u = x dt with |u| clamped to >= 1e-12; the reference applies the same clamp,
    so rows of tiny inputs are compared at their own scale.  Bars, and in brackets the worst element measured on a
    B200 (1000 W limit) as a fraction of its bar:
      true recurrence, every kernel   kappa = 2e-6   [0.44: 8.9e-7, scan_rp_kernel RP = 2 split, extreme inputs]
      quirk                           kappa = 2e-6   [0.27: 5.5e-7, 30,001 steps]
    The fp32 reference recurrence itself reaches 1.9e-7 of m (the quirk's streaming form 2.5e-7) under slow decay
    (test_oracle_fp32_within_bar): every kernel is within 5x of plain fp32 arithmetic, and the bars sit 5x below
    1e-5, which a kernel 20x less accurate than fp32 would still meet.
  * inputs: O(1) (dt = softplus(N(0, 1))), slow decay (dt log-uniform in [1e-3, 1e-1]: every state carries memory,
    so every power of the decay chains is visible), a trained-like spread of A for the generic kernels, and extremes
    placed across chunk boundaries (zero runs, 1e-25- and 1e4-scaled x, tiny, large, zero and denormal dt);
  * layouts: the model's (x | z interleaved, B | C | dt in one buffer) and padded strides, NaN in every gap and in
    the rows past B * L, a sentinel around y; the strided result equals the contiguous one bit for bit;
  * bit for bit: the row-packed shapes RP = 1 / 2, unsplit or split at any slot count, give the same bits; an
    utterance gives the same bits alone and in a batch; quirk rows do not depend on a CTA mate that never dies;
    a NaN in one (b, t, d) leaves every other row untouched;
  * long form (30,001 steps, slow dt): within the bar and within a small multiple of the fp32 reference's own error.
The CPU tests check the reference pieces: the magnitude bound, the clamp model, the quirk's streaming form.
VASR_ERR_LOG=<file> appends each comparison's worst fraction of its bar, for re-deriving the bars.
"""
import ctypes
import math
import os
import zlib
from ctypes import c_int32, c_int64, c_void_p

import numpy as np
import pytest

import velocity_oracle as O

gpu = pytest.mark.gpu

QUIRK, SEQ, RP = 1, 2, 3
OK, ERR_INVALID, ERR_SHAPE, ERR_UNSUPPORTED = 0, 1, 2, 5
KAPPA_TRUE = 2e-6
KAPPA_QUIRK = 2e-6
U_CLAMP = float(np.float32(1e-12))
TCH = 16                                   # timesteps per chunk of scan_seq_kernel / scan_rp_kernel (and the quirk's)
SENT = np.float32(-7777.25)
LS = (1, 7, 64, 203)                       # L = 1, below one chunk, a multiple of it, and with a partial last chunk


# ------------------------------------------------------------------ the variant table -----------
# (family, lpr, warps, rpl, structured, split): family 1 = scan_quirk_kernel<lpr, structured>, 2 =
# scan_seq_kernel<lpr, warps, rpl, structured>, 3 = scan_rp_kernel<RP = lpr, warps, OCC = rpl>; split: the launch is
# cut in time.  One entry per launch form launch_selective_scan can reach, read off its dispatch:
VARIANTS = ([(RP, rp, 4, occ, 1, sp) for rp, occ in ((1, 3), (2, 2)) for sp in (False, True)]       # rp_takes
            + [(SEQ, lpr, w, 2, st, False) for lpr, w in ((4, 4), (2, 4), (2, 2), (1, 2), (1, 1)) for st in (1, 0)]
            + [(QUIRK, lpr, 0, 0, st, False) for lpr in (8, 4, 2) for st in (1, 0)])


def vname(v):
    fam, lpr, w, rpl, st, sp = v
    if fam == RP:
        return f"rp{lpr}" + ("-split" if sp else "")
    if fam == SEQ:
        return f"seq{lpr}.{w}.{rpl}-" + ("S" if st else "G")
    return f"quirk{lpr}-" + ("S" if st else "G")


def spec(v, B=2):
    """How to reach v: N, Di, B, scan mode, A kind and the seam's override (rp, split, num_sms)."""
    fam, lpr, w, rpl, st, sp = v
    if fam == RP:
        return dict(N=64, Di=64 * lpr, B=3 if sp else B, quirk=0, structured=1, rp=lpr, split=0 if sp else -1,
                    num_sms=1 if sp else 0)
    if fam == SEQ:
        N = 16 * lpr
        Di = w * 2 * 32 // lpr
        return dict(N=N, Di=Di, B=B, quirk=0, structured=st, rp=-1, split=0, num_sms=0)
    return dict(N=8 * lpr, Di=64, B=B, quirk=1, structured=st, rp=0, split=0, num_sms=0)


def expect(v):
    """The variant the seam reports for v (slots aside)."""
    return tuple(v[:5])


def test_variant_table():
    assert len(VARIANTS) == 20
    assert len({v[:5] for v in VARIANTS}) == 18            # kernels: the split is a launch form of the same kernel
    for v in VARIANTS:
        s = spec(v)
        assert s["Di"] % 64 == 0


# ------------------------------------------------------------------ inputs ----------------------
def silu(z):
    return z / (1.0 + np.exp(-z))


def make_inputs(seed, B, L, Di, N, regime, structured, gate=True, skip=True):
    rng = np.random.default_rng(seed)
    f = np.float32
    x = rng.standard_normal((B, L, Di)).astype(f)
    if regime in ("o1", "extremes"):
        dt = np.log1p(np.exp(rng.standard_normal((B, L, Di)))).astype(f)
    else:                                                    # slow decay: log-uniform in [1e-3, 1e-1]
        dt = np.exp(rng.uniform(math.log(1e-3), math.log(1e-1), (B, L, Di))).astype(f)
    Bm = rng.standard_normal((B, L, N)).astype(f)
    Cm = rng.standard_normal((B, L, N)).astype(f)
    if structured:
        A = -np.arange(1, N + 1, dtype=f)
    elif regime == "trained":
        A = -np.exp(rng.uniform(-4.0, 2.0, N)).astype(f)
    else:
        A = -np.exp(rng.uniform(-1.0, 3.0, N)).astype(f)
    D = rng.standard_normal(Di).astype(f) if skip else None
    z = rng.standard_normal((B, L, Di)).astype(f) if gate else None
    if regime == "extremes":
        q = Di // 4
        x[:, 12:21, :q] = 0.0                                # a zero run across the first chunk boundary
        x[:, 30:35, q:2 * q] *= f(1e-25)                     # |u| far below the clamp, across the second
        x[:, 44:50, 2 * q:3 * q] *= f(1e4)                   # large, then back to O(1)
        dt[:, 14:18, 3 * q:] = f(1e-6)                       # decay ~ 1
        dt[:, 60:66, :2 * q] = f(20.0)                       # every state forgets
        dt[:, 95:96, :] = f(0.0)                             # a softplus that underflowed
        dt[:, 96:97, :] = f(1e-40)                           # denormal
        if B > 1:
            x[1, :, ::7] = 0.0                               # rows that are zero throughout
    return dict(x=x, dt=dt, A=A, Bm=Bm, Cm=Cm, D=D, z=z)


# ------------------------------------------------------------------ fp64 references --------------
def _f64(a):
    return None if a is None else np.asarray(a, np.float64)


def ref_true(inp, clamp):
    """The true recurrence in fp64 and the magnitude m of what it sums (module docstring).  clamp: |u| >= 1e-12 with
    its sign, as the structured kernels carry the state divided by u."""
    x, dt, A, Bm, Cm, D, z = (_f64(inp[k]) for k in ("x", "dt", "A", "Bm", "Cm", "D", "z"))
    Bsz, L, Di = x.shape
    h = np.zeros((Bsz, Di, A.size))
    ha = np.zeros_like(h)
    y = np.empty_like(x)
    m = np.empty_like(x)
    for t in range(L):
        dA = np.exp(dt[:, t, :, None] * A)
        u = x[:, t] * dt[:, t]
        if clamp:
            u = np.where(np.abs(u) < U_CLAMP, np.copysign(U_CLAMP, u), u)
        ub = u[..., None] * Bm[:, t, None, :]
        h = dA * h + ub
        ha = dA * ha + np.abs(ub)
        y[:, t] = np.einsum("bdn,bn->bd", h, Cm[:, t])
        m[:, t] = np.einsum("bdn,bn->bd", ha, np.abs(Cm[:, t]))
    y, m, _ = _skip_gate(x, D, z, y, m, np.zeros_like(m))
    return y, m


def ref_quirk(inp):
    """The reference's 'parallel' rule in its streaming form (velocity_oracle.scan_parallel_streaming) in fp64, with
    the magnitude of its terms carried alongside.  Returns (y, m, a): a is the part of m whose decay q = exp(A S) is
    below 2^-126, a term ex2.approx.ftz flushes to an exact zero (as does the reference's fp32 product of dA): the
    kernel may drop it whole, and its phases 2 / 3 rely on that."""
    x, dt, A, Bm, Cm, D, z = (_f64(inp[k]) for k in ("x", "dt", "A", "Bm", "Cm", "D", "z"))
    Bsz, L, Di = x.shape
    N = A.size
    H = np.zeros((Bsz, Di, N))
    Ha = np.zeros_like(H)
    S = np.zeros((Bsz, Di))
    nlev = max(1, L.bit_length() + 1)
    anc = [np.zeros((nlev, Bsz, Di, N)) for _ in range(5)]          # hP, H, |hP|, |H|, flushed part of |hP|
    anc_S = np.zeros((nlev, Bsz, Di))
    y = np.empty_like(x)
    m = np.empty_like(x)
    a = np.empty_like(x)
    aA = np.abs(A)
    for t in range(L):
        if t == 0:
            hp = np.zeros_like(H)
            hpa = np.zeros_like(H)
            hpf = np.zeros_like(H)
        else:
            lv = (t & -t).bit_length()
            php, pH, phpa, pHa, phpf, pS = (anc[0][lv], anc[1][lv], anc[2][lv], anc[3][lv], anc[4][lv],
                                            anc_S[lv])
            q = np.exp(A * S[..., None])
            pd = np.exp(A * (S - pS)[..., None])
            hp = php + q * (H - pd * pH)
            term = q * (1.0 + aA * S[..., None]) * (Ha + pd * pHa)
            hpa = phpa + term
            hpf = phpf + np.where(q < 2.0 ** -126, term, 0.0)
            for lvl in range(lv):
                anc[0][lvl], anc[1][lvl], anc[2][lvl], anc[3][lvl], anc[4][lvl] = hp, H, hpa, Ha, hpf
                anc_S[lvl] = S
        y[:, t] = np.einsum("bdn,bn->bd", hp, Cm[:, t])
        m[:, t] = np.einsum("bdn,bn->bd", hpa, np.abs(Cm[:, t]))
        a[:, t] = np.einsum("bdn,bn->bd", hpf, np.abs(Cm[:, t]))
        dA = np.exp(dt[:, t, :, None] * A)
        ub = (x[:, t] * dt[:, t])[..., None] * Bm[:, t, None, :]
        H = dA * H + ub
        Ha = dA * Ha + np.abs(ub)
        S = S + dt[:, t]
    return _skip_gate(x, D, z, y, m, a)


def _skip_gate(x, D, z, y, m, a):
    if D is not None:
        y = y + x * D
        m = m + np.abs(x * D)
    if z is not None:
        g = silu(z)
        y = y * g
        m = m * np.abs(g)
        a = a * np.abs(g)
    return y, m, a


def reference(v, inp):
    """(y, m, a): a = the flushed part of m the kernel may drop (ref_quirk), 0 for the true recurrence."""
    fam, st = v[0], v[4]
    if fam == QUIRK:
        return ref_quirk(inp)
    y, m = ref_true(inp, clamp=bool(st))
    return y, m, 0.0


def bar_fraction(got, ref, m, kappa, allow=0.0):
    """max over elements of |got - ref| / (kappa m + allow); an element with a zero bar must be exact."""
    err = np.abs(np.asarray(got, np.float64) - ref)
    bar = kappa * m + allow
    with np.errstate(divide="ignore", invalid="ignore"):
        frac = np.where(bar > 0, err / bar, np.where(err > 0, np.inf, 0.0))
    return float(frac.max()) if frac.size else 0.0, np.unravel_index(int(np.argmax(frac)), frac.shape)


def check(name, got, ref, m, kappa, allow=0.0):
    got = np.asarray(got)
    assert np.isfinite(got).all(), f"{name}: non-finite output"
    frac, where = bar_fraction(got, ref, m, kappa, allow)
    log = os.environ.get("VASR_ERR_LOG")
    if log:
        with open(log, "a") as f:
            f.write(f"{name}\t{frac * kappa:.3e}\t{frac:.4f}\n")
    assert frac <= 1.0, (f"{name}: (b, t, d) = {tuple(int(i) for i in where)}: |err| = "
                         f"{abs(float(got[where]) - ref[where]):.3e} > {kappa:.0e} x m = {kappa * m[where]:.3e}")


# ------------------------------------------------------------------ CPU checks of the reference ---
def test_oracle_fp32_within_bar():
    """The fp32 reference recurrence (velocity_oracle on float32 arrays) meets a quarter of the kernels' bar under
    slow decay, where error accumulates longest: the magnitude bound is not too tight for fp32 arithmetic."""
    inp = make_inputs(5, 2, 300, 64, 64, "slow", True)
    inp32 = dict(inp)
    y32 = O.scan_sequential(inp["x"], inp["dt"], inp["A"], inp["Bm"], inp["Cm"], inp["D"]) * silu(inp["z"])
    ref, m = ref_true(inp, clamp=False)
    assert bar_fraction(y32, ref, m, KAPPA_TRUE / 4)[0] <= 1.0
    yq = O.scan_parallel_streaming(inp32["x"], inp["dt"], inp["A"], inp["Bm"], inp["Cm"], inp["D"]) * silu(inp["z"])
    refq, mq, aq = ref_quirk(inp)
    assert bar_fraction(yq, refq, mq, KAPPA_QUIRK / 4, aq)[0] <= 1.0


def test_reference_matches_oracle():
    """ref_true / ref_quirk without clamp equal the oracle's fp64 scans; the quirk's also the literal tree scan."""
    inp = make_inputs(6, 2, 37, 64, 16, "o1", False)
    d = {k: _f64(v) for k, v in inp.items()}
    y, _ = ref_true(inp, clamp=False)
    want = O.scan_sequential(d["x"], d["dt"], d["A"], d["Bm"], d["Cm"], d["D"]) * silu(d["z"])
    np.testing.assert_allclose(y, want, rtol=1e-12, atol=1e-12)
    yq, _, _ = ref_quirk(inp)
    want_q = O.scan_parallel(d["x"], d["dt"], d["A"], d["Bm"], d["Cm"], d["D"]) * silu(d["z"])
    np.testing.assert_allclose(yq, want_q, rtol=1e-9, atol=1e-9)


def test_clamp_model():
    """The clamp changes nothing where |u| >= 1e-12, and elsewhere moves y by at most the clamp's own terms."""
    inp = make_inputs(7, 2, 60, 64, 64, "extremes", True)
    y0, m0 = ref_true(inp, clamp=False)
    y1, m1 = ref_true(inp, clamp=True)
    u = np.abs(inp["x"].astype(np.float64) * inp["dt"])
    tiny_rows = (u < U_CLAMP).any(axis=1)                    # (B, Di): rows with a clamped step
    assert tiny_rows.any() and (~tiny_rows).any()
    b, d = np.nonzero(~tiny_rows)
    assert np.array_equal(y0[b, :, d], y1[b, :, d])
    # elsewhere: each clamped step adds at most 1e-12 |B| to a state whose decay is <= 1
    bound = U_CLAMP * np.abs(inp["Bm"]).sum(-1).max() * np.abs(inp["Cm"]).sum(-1).max() * 60
    assert np.abs(y1 - y0).max() <= bound * np.abs(silu(inp["z"].astype(np.float64))).max()


def test_magnitude_bounds_the_result():
    """|y| <= m for both references (m is a bound on what the output sums, so the bar is relative to it)."""
    for regime in ("o1", "slow", "extremes"):
        inp = make_inputs(8, 2, 100, 64, 32, regime, True)
        for y, m in (ref_true(inp, clamp=True), ref_quirk(inp)[:2]):
            assert (np.abs(y) <= m * (1 + 1e-12) + 1e-300).all(), regime


def cut_positions(total_chunks, slots, cpc):
    """(chain, chunk within it) where each slot after the first begins, as scan_rp_kernel deals the chunks out."""
    return [divmod(total_chunks * s // slots, cpc) for s in range(1, slots)]


def test_cut_positions():
    assert cut_positions(30, 6, 3) == [(1, 2), (3, 1), (5, 0), (6, 2), (8, 1)]


# ------------------------------------------------------------------ the seam (GPU) --------------
class _ScanCall(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("ldx", c_int64), ("dt", c_void_p), ("lddt", c_int64), ("z", c_void_p),
                ("ldz", c_int64), ("Bm", c_void_p), ("ldb", c_int64), ("Cm", c_void_p), ("ldc", c_int64),
                ("A", c_void_p), ("D", c_void_p), ("y", c_void_p), ("ldy", c_int64), ("B", c_int64), ("L", c_int64),
                ("Di", c_int32), ("N", c_int32), ("parallel_quirk", c_int32), ("structured", c_int32),
                ("num_sms", c_int32), ("rp", c_int32), ("split", c_int32), ("stream", c_void_p),
                ("variant", c_int32 * 6)]


@pytest.fixture(scope="module")
def torch():
    import torch as t
    assert t.cuda.is_available(), "GPU tests need a CUDA device"
    return t


@pytest.fixture(scope="module")
def seam(torch):
    from velocity_asr import _native
    fn = _native.lib().vasr_debug_scan
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.POINTER(_ScanCall)]
    return fn


def _buf(torch, rows, ld, fill):
    return torch.full((rows, ld), float(fill), dtype=torch.float32, device="cuda")


def run(torch, seam, inp, s, layout="contig", **over):
    """One seam call.  Returns (rc, y (B, L, Di) float32 or None, variant tuple).  The layouts put every input in a
    buffer with NaN in its gaps and in PAD rows past B * L, and y between sentinel rows (and in sentinel gaps)."""
    o = dict(s)
    o.update(over)
    x, dt, z, Bm, Cm = inp["x"], inp["dt"], inp["z"], inp["Bm"], inp["Cm"]
    Bsz, L, Di = x.shape
    N = Bm.shape[-1]
    M, PAD = Bsz * L, 3
    nan = float("nan")
    keep = []

    def put(a, ld, off=0, shift=0):
        t = torch.full(((M + PAD) * ld + shift + 4,), nan, dtype=torch.float32, device="cuda")
        if a is not None:
            t[shift:shift + M * ld].view(M, ld)[:, off:off + a.shape[-1]] = torch.from_numpy(a.reshape(M, -1)).cuda()
        keep.append(t)
        return t[shift:].data_ptr() + 4 * off

    if layout == "contig":
        px, lx = put(x, Di), Di
        pd, ld = put(dt, Di), Di
        pz, lz = (put(z, Di), Di) if z is not None else (None, Di)
        pb, lb = put(Bm, N), N
        pc, lc = put(Cm, N), N
        ly, yshift = Di, 0
    elif layout == "model":                                  # x | z and B | C | dt, as run_scan passes them
        xz = np.concatenate([x, z if z is not None else np.zeros_like(x)], -1)
        bcdt = np.concatenate([Bm, Cm, dt], -1)
        base_xz = put(xz, 2 * Di)
        base_bc = put(bcdt, 2 * N + Di)
        px, lx = base_xz, 2 * Di
        pz, lz = (base_xz + 4 * Di, 2 * Di) if z is not None else (None, 2 * Di)
        pb, lb = base_bc, 2 * N + Di
        pc, lc = base_bc + 4 * N, 2 * N + Di
        pd, ld = base_bc + 8 * N, 2 * N + Di
        ly, yshift = Di, 0
    elif layout == "padded":
        px, lx = put(x, Di + 8, off=4), Di + 8
        pd, ld = put(dt, Di + 4), Di + 4
        pz, lz = (put(z, Di + 12, off=8), Di + 12) if z is not None else (None, 0)
        pb, lb = put(Bm, N + 4), N + 4
        pc, lc = put(Cm, N + 8, off=4), N + 8
        ly, yshift = Di + 8, 0
    elif layout == "odd":                                    # rows that are not 16-byte aligned (no cp.async)
        if o["quirk"]:
            px, lx = put(x, Di + 1, shift=1), Di + 1
            pd, ld = put(dt, Di + 3, shift=3), Di + 3
            pz, lz = (put(z, Di + 1, shift=2), Di + 1) if z is not None else (None, 0)
            ly, yshift = Di + 1, 1
        else:                                                # scan_seq_kernel: y rows 8-byte aligned only
            px, lx = put(x, Di), Di
            pd, ld = put(dt, Di), Di
            pz, lz = (put(z, Di), Di) if z is not None else (None, 0)
            ly, yshift = Di + 2, 2
        pb, lb = put(Bm, N), N
        pc, lc = put(Cm, N), N
    else:
        raise ValueError(layout)
    A = torch.from_numpy(inp["A"]).cuda()
    D = torch.from_numpy(inp["D"]).cuda() if inp["D"] is not None else None
    ybuf = torch.full(((M + 2) * ly + yshift + 4,), float(SENT), dtype=torch.float32, device="cuda")
    a = _ScanCall()
    a.x, a.ldx, a.dt, a.lddt, a.z, a.ldz = px, lx, pd, ld, pz, lz
    a.Bm, a.ldb, a.Cm, a.ldc = pb, lb, pc, lc
    a.A, a.D = A.data_ptr(), (D.data_ptr() if D is not None else None)
    a.y, a.ldy = ybuf.data_ptr() + 4 * (yshift + ly), ly
    a.B, a.L, a.Di, a.N = Bsz, L, Di, N
    a.parallel_quirk, a.structured = o["quirk"], o["structured"]
    a.num_sms, a.rp, a.split = o["num_sms"], o["rp"], o["split"]
    a.stream = torch.cuda.current_stream().cuda_stream
    rc = seam(ctypes.byref(a))
    var = tuple(a.variant)
    if rc != OK:
        return rc, None, var
    yb = ybuf.cpu().numpy()
    body = yb[yshift + ly:yshift + ly + M * ly].reshape(M, ly)
    assert (yb[:yshift + ly] == SENT).all() and (yb[yshift + ly + M * ly:] == SENT).all(), "write outside y's rows"
    assert (body[:, Di:] == SENT).all(), "write into y's row gaps"
    return rc, body[:, :Di].reshape(Bsz, L, Di).copy(), var


def run_ok(torch, seam, inp, s, v, layout="contig", **over):
    rc, y, var = run(torch, seam, inp, s, layout, **over)
    assert rc == OK, f"{vname(v)}: vasr_debug_scan returned {rc}"
    assert var[:5] == expect(v), f"{vname(v)}: launched {var}"
    if v[0] == RP and "num_sms" not in over and "rp" not in over and "split" not in over:
        assert (var[5] > 0) == v[5], f"{vname(v)}: slots {var[5]}"
    return y, var


def kappa(v):
    return KAPPA_QUIRK if v[0] == QUIRK else KAPPA_TRUE


def _regimes(v):
    return ("o1", "slow", "extremes") + (("trained",) if not v[4] else ())


CASES = [pytest.param(v, r, id=f"{vname(v)}-{r}") for v in VARIANTS for r in _regimes(v)]


@gpu
def test_variant_coverage(torch, seam):
    """Every launch form of the table is reached by its spec, and nothing else is reported."""
    seen = set()
    for v in VARIANTS:
        s = spec(v)
        inp = make_inputs(1, s["B"], 40, s["Di"], s["N"], "o1", s["structured"])
        _, var = run_ok(torch, seam, inp, s, v)
        seen.add(var[:5] + (var[5] > 0,))
    assert seen == set(VARIANTS)


@gpu
@pytest.mark.parametrize("v,regime", CASES)
def test_scan_variant(torch, seam, v, regime):
    s = spec(v)
    for i, L in enumerate(LS):
        gate, skip = (i % 2 == 0), (i != 1)                  # without gate and without skip too
        inp = make_inputs(zlib.crc32(f"{vname(v)} {regime} {L}".encode()), s["B"], L, s["Di"], s["N"], regime, s["structured"],
                          gate=gate, skip=skip)
        y, _ = run_ok(torch, seam, inp, s, v)
        ref, m, a = reference(v, inp)
        check(f"{vname(v)} {regime} L={L}", y, ref, m, kappa(v), a)


def _layouts(v):
    return ("model", "padded") + (("odd",) if v[0] != RP else ())


@gpu
@pytest.mark.parametrize("v,layout", [pytest.param(v, lay, id=f"{vname(v)}-{lay}") for v in VARIANTS
                                      for lay in _layouts(v)])
def test_layout_and_fences(torch, seam, v, layout):
    """Strided inputs with NaN in every gap and past the last row, y between sentinels: the same bits as contiguous."""
    s = spec(v)
    for gate in (True, False):
        inp = make_inputs(11, s["B"], 45, s["Di"], s["N"], "o1", s["structured"], gate=gate)
        want, var0 = run_ok(torch, seam, inp, s, v)
        got, var1 = run_ok(torch, seam, inp, s, v, layout=layout)
        assert var0 == var1
        assert np.array_equal(got, want), f"{vname(v)} {layout}: differs from the contiguous run"


@gpu
def test_rp_rejects_unaligned_rows(torch, seam):
    s = spec(VARIANTS[0])
    inp = make_inputs(2, 2, 20, 64, 64, "o1", True)
    rc, _, var = run(torch, seam, inp, s, layout="odd", quirk=0, rp=1)
    assert rc == ERR_UNSUPPORTED and var == (0,) * 6


# ------------------------------------------------------------------ bit-for-bit invariants -------
@gpu
def test_rp_shapes_and_splits_same_bits(torch, seam):
    """scan_rp_kernel RP = 1 and RP = 2, unsplit and split at several SM counts, give identical bits.  5 x 45 steps
    x 128 rows: 3 chunks per chain (the last one partial); the cuts fall at chain starts, mid-chain and in the last
    partial chunk (checked from the reported slot counts)."""
    Bsz, L, Di = 5, 45, 128
    inp = make_inputs(21, Bsz, L, Di, 64, "slow", True)
    s = spec(VARIANTS[0])
    base, _ = run_ok(torch, seam, inp, s, VARIANTS[0], rp=1, split=-1)
    dev_sms = torch.cuda.get_device_properties(0).multi_processor_count
    cpc = (L + TCH - 1) // TCH
    kinds = set()
    for rp in (1, 2):
        for sms in (1, 2, 3, 5, 7, dev_sms):
            rc, y, var = run(torch, seam, inp, s, rp=rp, split=0, num_sms=sms)
            assert rc == OK and var[:2] == (RP, rp)
            assert np.array_equal(y, base), f"RP = {rp}, {sms} SMs ({var[5]} slots): bits differ"
            if var[5]:
                chains = Bsz * Di // (64 * rp)
                for _, k in cut_positions(chains * cpc, var[5], cpc):
                    kinds.add("start" if k == 0 else ("last partial" if k == cpc - 1 else "mid"))
    assert kinds == {"start", "mid", "last partial"}, kinds


@gpu
@pytest.mark.parametrize("v", [pytest.param(v, id=vname(v)) for v in VARIANTS])
def test_alone_equals_in_batch(torch, seam, v):
    """Utterance 1 of a batch of 3 (of 5 for the split forms) gets the bits it gets alone."""
    s = spec(v, B=3)
    Bsz = 5 if v[5] else 3
    inp = make_inputs(31, Bsz, 50, s["Di"], s["N"], "slow", s["structured"])
    s["B"] = Bsz
    batch, _ = run_ok(torch, seam, inp, s, v)
    one = {k: (a[1:2].copy() if a is not None and a.ndim == 3 else a) for k, a in inp.items()}
    rc, alone, var = run(torch, seam, one, s)
    assert rc == OK and var[:5] == expect(v)
    assert np.array_equal(alone[0], batch[1])


@gpu
@pytest.mark.parametrize("v", [pytest.param(v, id=vname(v)) for v in VARIANTS])
def test_nan_stays_in_its_row(torch, seam, v):
    s = spec(v)
    inp = make_inputs(41, s["B"], 70, s["Di"], s["N"], "o1", s["structured"])
    clean, _ = run_ok(torch, seam, inp, s, v)
    b0, t0, d0 = s["B"] - 1, 23, 5
    bad = dict(inp)
    bad["x"] = inp["x"].copy()
    bad["x"][b0, t0, d0] = np.nan
    got, _ = run_ok(torch, seam, bad, s, v)
    mask = np.ones(got.shape, bool)
    mask[b0, t0:, d0] = False
    assert np.array_equal(got[mask], clean[mask])
    assert np.isnan(got[b0, t0, d0])


@gpu
@pytest.mark.parametrize("v", [pytest.param(v, id=vname(v)) for v in VARIANTS if v[0] == QUIRK])
def test_quirk_rows_do_not_depend_on_cta_mates(torch, seam, v):
    """Phases 2 / 3 are shortcuts of the full rule: a row gets the same bits next to a CTA mate that never dies and so
    keeps its CTA in phase 1.  Without the D skip, y past the switch is the bare sum of the flushed terms, so a switch
    before they are exact zeros shows as bits (and against the reference, whose terms above 2^-126 the kernel must
    keep).  With structured A the mate follows its CTA into the narrow mode (same dt until t = 64) and stops decaying
    after: the narrow mode drops only exact zeros too, but it computes the kept states' powers and sums them in
    another order than the wide mode, so the last bit of a row's state sum depends on when its CTA narrows."""
    s = spec(v)
    rows = 128 // v[1]
    L = 300
    for skip in (True, False):
        inp = make_inputs(51, s["B"], L, s["Di"], s["N"], "o1", s["structured"], skip=skip)
        if not s["structured"]:
            inp["A"] = -np.exp(np.random.default_rng(3).uniform(-0.5, 3.0, s["N"])).astype(np.float32)
        inp["dt"][:, :, rows // 2:rows] *= np.float32(0.3)    # rows of a CTA that die later than their mates
        alone, _ = run_ok(torch, seam, inp, s, v)
        mate = dict(inp)
        mate["dt"] = inp["dt"].copy()
        mate["dt"][:, 64 if s["structured"] else 0:, ::rows] *= np.float32(1e-3)    # one row per CTA never dies
        got, _ = run_ok(torch, seam, mate, s, v)
        keep = np.ones(s["Di"], bool)
        keep[::rows] = False
        assert np.array_equal(got[:, :, keep], alone[:, :, keep]), f"skip {skip}"
        ref, m, a = ref_quirk(inp)
        check(f"{vname(v)} phases skip={skip}", alone, ref, m, KAPPA_QUIRK, a)


# ------------------------------------------------------------------ long form --------------------
def _long_inputs(N, structured, dt_lo, dt_hi, seed):
    rng = np.random.default_rng(seed)
    L, Di = 30001, 64
    f = np.float32
    inp = dict(x=rng.standard_normal((1, L, Di)).astype(f),
               dt=np.exp(rng.uniform(math.log(dt_lo), math.log(dt_hi), (1, L, Di))).astype(f),
               Bm=rng.standard_normal((1, L, N)).astype(f), Cm=rng.standard_normal((1, L, N)).astype(f),
               A=(-np.arange(1, N + 1, dtype=f) if structured else -np.exp(rng.uniform(-4.0, 2.0, N)).astype(f)),
               D=rng.standard_normal(Di).astype(f), z=rng.standard_normal((1, L, Di)).astype(f))
    return inp


def _row_rel(got, ref):
    return float((np.abs(np.asarray(got, np.float64) - ref).max(axis=1) / np.abs(ref).max(axis=1)).max())


LONG_MULT = 5          # measured: 1.8x (rp), 2.1x (generic seq), 2.5x (quirk) the fp32 reference's error


@gpu
@pytest.mark.parametrize("v,dt_lo,dt_hi", [
    pytest.param(VARIANTS[0], 1e-3, 1e-1, id="rp1"),
    pytest.param((SEQ, 4, 4, 2, 0, False), 1e-3, 1e-1, id="seq4.4.2-G"),
    pytest.param((QUIRK, 8, 0, 0, 1, False), 1e-4, 5e-3, id="quirk8-S"),        # sum dt ~ 38: phase 1 throughout
])
def test_long_form(torch, seam, v, dt_lo, dt_hi):
    """Config 4's length (one 600 s utterance = 30,001 tokens) with slow dt: within the bar, and within LONG_MULT
    times the fp32 reference recurrence's own error (row-relative) on the same inputs."""
    s = spec(v, B=1)
    inp = _long_inputs(s["N"], s["structured"], dt_lo, dt_hi, 61)
    y, _ = run_ok(torch, seam, inp, s, v)
    ref, m, a = reference(v, inp)
    check(f"{vname(v)} L=30001", y, ref, m, kappa(v), a)
    if v[0] == QUIRK:
        assert float(inp["dt"].astype(np.float64).sum(axis=1).max()) * 1.4427 < 127      # never dead: phase 1
        y32 = O.scan_parallel_streaming(inp["x"], inp["dt"], inp["A"], inp["Bm"], inp["Cm"], inp["D"])
    else:
        y32 = O.scan_sequential(inp["x"], inp["dt"], inp["A"], inp["Bm"], inp["Cm"], inp["D"])
    y32 = y32 * silu(inp["z"])
    e_kernel, e32 = _row_rel(y, ref), _row_rel(y32, ref)
    log = os.environ.get("VASR_ERR_LOG")
    if log:
        with open(log, "a") as f:
            f.write(f"{vname(v)} long: kernel {e_kernel:.3e} fp32 reference {e32:.3e}\n")
    assert e_kernel <= LONG_MULT * e32, f"{vname(v)}: {e_kernel:.2e} against the fp32 reference's {e32:.2e}"


# ------------------------------------------------------------------ A detection, contract ---------
@gpu
@pytest.mark.parametrize("rel,structured", [(1.5e-6, True), (3e-6, False)])
def test_structured_detection_boundary(torch, seam, rel, structured):
    """A = -(n + 1)(1 +- rel), alternating: within 2e-6 the structured kernel, beyond it the generic one; each
    within the bar computed with the A given."""
    N, Di = 64, 64
    inp = make_inputs(71, 2, 203, Di, N, "slow", True)
    sign = np.where(np.arange(N) % 2 == 0, 1.0, -1.0)
    inp["A"] = (-(np.arange(1, N + 1)) * (1.0 + sign * rel)).astype(np.float32)
    s = dict(N=N, Di=Di, B=2, quirk=0, structured=-1, rp=0, split=-1, num_sms=0)
    rc, y, var = run(torch, seam, inp, s)
    assert rc == OK
    assert var[0] == (RP if structured else SEQ) and var[4] == int(structured), var
    ref, m = ref_true(inp, clamp=structured)
    check(f"A rel {rel}", y, ref, m, KAPPA_TRUE)


@gpu
def test_seam_refusals(torch, seam):
    inp = make_inputs(81, 1, 20, 64, 64, "o1", False)
    s = dict(N=64, Di=64, B=1, quirk=0, structured=1, rp=0, split=0, num_sms=0)
    assert run(torch, seam, inp, s)[0] == ERR_INVALID                          # "structured" for an A that is not
    inp = make_inputs(81, 1, 20, 64, 64, "o1", True)
    dev_sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert run(torch, seam, inp, s, num_sms=dev_sms + 1)[0] == ERR_INVALID     # more SMs than the device has
    assert run(torch, seam, inp, s, split=3)[0] == ERR_INVALID                 # slot counts only through num_sms
    assert run(torch, seam, inp, s, rp=2)[0] == ERR_UNSUPPORTED                # RP = 2 needs 128-row chains
    rc, _, var = run(torch, seam, inp, s, structured=0)
    assert rc == OK and var[:5] == (SEQ, 4, 4, 2, 0)                           # the generic kernel on any A


@gpu
@pytest.mark.parametrize("Di", [48, 96, 32])
def test_di_must_be_a_multiple_of_64(torch, Di):
    import velocity_asr as va
    from velocity_asr import _native
    x = torch.zeros(1, 4, Di, device="cuda")
    A = -torch.arange(1, 65, device="cuda", dtype=torch.float32)
    Bm = torch.zeros(1, 4, 64, device="cuda")
    with pytest.raises(ValueError):
        va.selective_scan(x, x, A, Bm, Bm, scan_mode="sequential")
    y = torch.empty_like(x)
    p = _native.ptr
    rc = _native.lib().vasr_selective_scan(p(x), Di, p(x), Di, p(A), p(Bm), 64, p(Bm), 64, None, None, Di, p(y), Di,
                                           1, 4, Di, 64, 0, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == ERR_SHAPE
