"""The operand format of the tensor-core projection (csrc/gemm_tc.cu): TF32 hi words and paired-bf16 correction words.

`vasr_split_tf32` leaves W as (2, N, K) 32-bit words: hi = rna_tf32(w) and, per element, the pair
(bf16(hi), bf16(w - hi)) in the low and high half of one word.  The converters pack each activation x as
(bf16(x - hi), bf16(hi)), so one kind::f16 MMA over the pair words computes A_lo·W_hi + A_hi·W_lo and one kind::tf32
MMA adds A_hi·W_hi.
  * the split buffer equals a numpy emulation bit for bit (rna TF32: ties away from zero; bf16: round to nearest
    even), on ±0, subnormals, exact bf16 ties of hi and of w - hi, and K = 4 / 36 / 240;
  * at the projection shapes of the model (tools/gemm_bench.py) with M = 12,016 rows, every row's error against an
    fp64 reference stays within 3e-6 of the row's max |pre-activation| (or |output| where that is larger).  A lost
    correction term costs about 2^-12 and halves swapped between A and W pair A_lo with W_lo (about 2^-9).
"""
import numpy as np
import pytest
import torch

import velocity_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def va():
    import velocity_asr
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return velocity_asr


def rna_tf32_bits(x):
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x1000) & 0xFFFFE000).astype(np.uint32)


def rn_bf16_bits(x):
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint32)


def split_emulated(w):
    hi = rna_tf32_bits(w)
    hif = hi.view(np.float32)
    lo = w - hif                                           # exact: the residual of a rounding to 11 bits
    return np.stack([hi, (rn_bf16_bits(lo) << 16) | rn_bf16_bits(hif)])


def awkward_weights(N, K, seed):
    """Random values with ±0, subnormals and exact bf16 ties of hi and of w - hi mixed in."""
    rng = np.random.default_rng(seed)
    w = (rng.standard_normal((N, K)) * np.exp2(rng.integers(-20, 20, (N, K)))).astype(np.float32)
    flat = w.reshape(-1)
    n = flat.size
    pick = rng.permutation(n)
    q = max(n // 8, 1)
    sub = (rng.integers(1, 1 << 23, q) * rng.choice([1, -1], q)).astype(np.int64)
    flat[pick[:q]] = np.abs(sub).astype(np.uint32).view(np.float32) * np.sign(sub).astype(np.float32)
    # hi on a bf16 tie: low 16 bits of a TF32 value exactly 0x8000, both parities of the kept bit
    hb = (rng.integers(0x3C00, 0x4400, q).astype(np.uint32) << 16) | 0x8000
    flat[pick[q:2 * q]] = hb.view(np.float32) * rng.choice([1, -1], q).astype(np.float32)
    # w - hi on a bf16 tie: hi a TF32 value, the residual a value with low 16 bits 0x8000 below half its ulp
    hi = (rng.integers(0x3C00, 0x4400, q).astype(np.uint32) << 16) | (rng.integers(0, 8, q).astype(np.uint32) << 13)
    lo = ((hi & 0x7F800000) - (14 << 23)) | (rng.integers(0, 0x7F, q).astype(np.uint32) << 16) | 0x8000
    r = hi.view(np.float32) + lo.view(np.float32) * rng.choice([1, -1], q).astype(np.float32)
    flat[pick[2 * q:3 * q]] = r
    flat[pick[3 * q]] = 0.0
    flat[pick[3 * q + 1]] = -0.0
    return w


@pytest.mark.parametrize("K", [4, 36, 240])
def test_split_buffer_matches_emulation(va, K):
    w = awkward_weights(48, K, seed=K)
    got = va.split_tf32(torch.from_numpy(w).cuda()).cpu().numpy().view(np.uint32)
    want = split_emulated(w)
    assert got.shape == want.shape == (2, 48, K)
    bad = np.argwhere(got != want)
    assert bad.size == 0, (f"{len(bad)} words differ; first at {tuple(bad[0])}: w = {w[tuple(bad[0][1:])]!r}, "
                           f"got {got[tuple(bad[0])]:#010x}, want {want[tuple(bad[0])]:#010x}")


# (name, K, N, activation, residual) of tools/gemm_bench.py
SHAPES = [("in_proj", 192, 768, None, False), ("x_dt_proj", 384, 512, "softplus", False),
          ("out_proj", 384, 192, None, True), ("ffn1", 192, 384, "gelu", False), ("ffn2", 384, 192, None, True),
          ("ctc", 192, 1000, None, False), ("fusion3", 384, 576, None, False)]
ACT = {None: lambda v: v, "gelu": O.gelu, "softplus": O.softplus}


@pytest.mark.parametrize("name,K,N,act,resid", SHAPES, ids=[s[0] for s in SHAPES])
def test_projection_error_at_model_shapes(va, name, K, N, act, resid):
    M = 12016
    rng = np.random.default_rng(K * 7919 + N)
    x = rng.standard_normal((M, K)).astype(np.float32)
    w = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    r = rng.standard_normal((M, N)).astype(np.float32) if resid else None
    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()
    wd = dev(w)
    out = va.linear(dev(x), wd, dev(b), activation=act, tensor_cores=True, weight_split=va.split_tf32(wd),
                    residual=dev(r)).cpu().numpy().astype(np.float64)
    pre = x.astype(np.float64) @ w.T.astype(np.float64) + b
    ref = ACT[act](pre) + (r if resid else 0.0)
    scale = np.maximum(np.abs(pre).max(axis=1), np.abs(ref).max(axis=1))
    err = (np.abs(out - ref).max(axis=1) / scale).max()
    assert err <= 3e-6, f"{name}: worst row error {err:.3g} of the row max"
