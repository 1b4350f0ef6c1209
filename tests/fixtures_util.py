"""Seeded inputs shared by the golden generator (build container) and the tests (any box)."""
import numpy as np
import torch

AUDIO_SEED = 1234     # SURVEY.md section 8(d)
WEIGHT_SEED = 0


def synth_audio(batch: int, samples: int, seed: int = AUDIO_SEED) -> torch.Tensor:
    """Broadband Gaussian PCM, sigma 0.1 (tonal input makes the fp32 reference itself noisy)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(batch, samples, generator=g) * 0.1


def amplify_state_dict(sd: dict, seed: int = 7) -> dict:
    """Deterministic re-scaling of a random-init state dict so that the SSM branch is
    numerically visible at the logits (at plain random init it is ~2e-3 of the residual
    stream, SURVEY.md section 0 item 5) and A is no longer exactly -(1..N)."""
    rs = np.random.RandomState(seed)
    out = {}
    for k, v in sd.items():
        v = v.clone()
        if k.endswith("ssm.A_log"):
            v += torch.from_numpy(rs.uniform(-0.4, 0.4, size=tuple(v.shape)).astype(np.float32))
        elif k.endswith("ssm.D"):
            v = torch.from_numpy(rs.standard_normal(tuple(v.shape)).astype(np.float32))
        elif k.endswith("ssm.dt_proj.bias"):
            v = torch.from_numpy(rs.uniform(-3.0, 0.0, size=tuple(v.shape)).astype(np.float32))
        elif k.endswith("ssm.out_proj.weight"):
            v *= 6.0
        elif k.endswith("ssm.x_proj.weight"):
            v *= 3.0
        elif k.endswith(".conv.weight") and "layers" in k:
            v *= 3.0
        out[k] = v
    return out


def scan_inputs(batch, length, d_inner, n_state, seed, structured_a=True):
    """O(1) per-op scan inputs (SURVEY.md section 8(d)): x,B,C ~ N(0,1), dt = softplus(N(0,1))."""
    rs = np.random.RandomState(seed)
    x = rs.standard_normal((batch, length, d_inner)).astype(np.float32)
    dt = np.log1p(np.exp(rs.standard_normal((batch, length, d_inner)))).astype(np.float32)
    Bm = rs.standard_normal((batch, length, n_state)).astype(np.float32)
    Cm = rs.standard_normal((batch, length, n_state)).astype(np.float32)
    D = rs.standard_normal(d_inner).astype(np.float32)
    if structured_a:
        A = -np.exp(np.log(np.arange(1, n_state + 1, dtype=np.float32))).astype(np.float32)
    else:
        A = -np.exp(rs.uniform(-1.0, 3.0, size=n_state)).astype(np.float32)
    return x, dt, A, Bm, Cm, D


def state_dict_digest(sd: dict) -> np.ndarray:
    """(n_tensors, 2) float64: sum and abs-sum per tensor in key order — proves two boxes
    drew the same random init without shipping 25 MB of weights."""
    return np.array([[float(v.double().sum()), float(v.double().abs().sum())] for _, v in sd.items()])


def state_dict_fingerprint(sd: dict) -> list:
    """'<key> <shape> <sha256 of the bytes>' per tensor in key order: equal lists mean equal trees, bit for bit."""
    import hashlib
    return [f"{k} {tuple(v.shape)} {hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest()}"
            for k, v in sd.items()]
