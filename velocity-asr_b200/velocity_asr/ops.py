"""Operator-level entry points: the selective scan behind the reference's scan_mode switch
(velocity_asr/ssm.py:119-126) and a plain linear layer, both through the C ABI."""
import ctypes
from typing import Optional

import torch

from . import _native


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _f32c(t):
    return None if t is None else t.to(torch.float32).contiguous()


def selective_scan(x: torch.Tensor, dt: torch.Tensor, A: torch.Tensor, B: torch.Tensor, C: torch.Tensor,
                   D: Optional[torch.Tensor] = None, z: Optional[torch.Tensor] = None,
                   scan_mode: str = "sequential", validate: bool = True) -> torch.Tensor:
    """x, dt: (B, L, Di); A: (N,); B, C: (B, L, N); D: (Di,) -> y (B, L, Di).

    scan_mode 'sequential' / 'mamba' = SelectiveSSM._sequential_scan (ssm.py:134-171);
    'parallel' = _parallel_scan exactly as shipped (ssm.py:173-295).  With z given, the result is
    y * silu(z) (ssm.py:129).  N in {16, 32, 64}; Di a multiple of 64.  validate=False skips the (synchronising)
    check that dt is non-negative in 'parallel' mode."""
    if scan_mode not in _native.SCAN_MODE_ID:
        raise ValueError(f"Unknown scan_mode: {scan_mode}")
    if x.device.type != "cuda":
        raise RuntimeError("selective_scan runs on CUDA only (no CPU fallback)")
    x, dt, A, B, C, D, z = map(_f32c, (x, dt, A, B, C, D, z))
    if validate and scan_mode == "parallel" and dt.numel() and bool((dt < 0).any()):
        # the 'parallel' kernel stops evaluating terms once exp(A * cumsum(dt)) has decayed to an exact zero, which
        # presumes a growing cumsum: dt is a softplus output wherever the reference calls its scan (ssm.py:118)
        raise ValueError("selective_scan(scan_mode='parallel') needs dt >= 0 (dt is a softplus output, ssm.py:118)")
    Bsz, L, Di = x.shape
    if Di <= 0 or Di % 64 != 0:
        raise ValueError(f"selective_scan needs Di to be a positive multiple of 64, got {Di}")
    N = A.numel()
    y = torch.empty_like(x)
    if Bsz == 0 or L == 0:
        return y
    lib = _native.lib()
    with torch.cuda.device(x.device):
        _native.check(lib.vasr_selective_scan(
            _native.ptr(x), Di, _native.ptr(dt), Di, _native.ptr(A), _native.ptr(B), N, _native.ptr(C), N,
            _native.ptr(D), _native.ptr(z), Di, _native.ptr(y), Di, Bsz, L, Di, N,
            _native.SCAN_MODE_ID[scan_mode], _stream(x.device)))
    return y


def selective_scan_fn(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False,
                      return_last_state=False):
    """Signature of mamba_ssm.ops.selective_scan_interface.selective_scan_fn as the reference
    calls it (ssm.py:326-332): u, delta (B, D, L); A (D, N) with identical rows; B, C (B, 1, L, N);
    D (D,) -> (B, D, L)."""
    if delta_bias is not None or delta_softplus or return_last_state or z is not None:
        raise NotImplementedError("only the call pattern of velocity_asr/ssm.py:326-332 is supported")
    if not bool((A == A[:1]).all()):
        raise NotImplementedError("A must be shared by all channels (ssm.py:317)")
    y = selective_scan(u.transpose(1, 2), delta.transpose(1, 2), A[0], B.squeeze(1), C.squeeze(1), D,
                       scan_mode="mamba")
    return y.transpose(1, 2).contiguous()


_ACT = {None: 0, "none": 0, "gelu": 1, "softplus": 2, "sigmoid": 3}


def split_tf32(weight: torch.Tensor) -> torch.Tensor:
    """(N, K) fp32 weight -> (2, N, K) 32-bit words, the operand format of the tensor-core projection kernel:
    [0] = rna_tf32(w) (float32), [1] = a pair of bf16 per word, bf16(hi) in the low and bf16(w - hi) in the high
    16 bits (view as int32 / uint32 to read them).  Done once per weight matrix."""
    if weight.device.type != "cuda":
        raise RuntimeError("split_tf32 runs on CUDA only (no CPU fallback)")
    weight = _f32c(weight)
    out = torch.empty((2,) + tuple(weight.shape), device=weight.device, dtype=torch.float32)
    with torch.cuda.device(weight.device):
        _native.check(_native.lib().vasr_split_tf32(_native.ptr(weight), _native.ptr(out), weight.numel(),
                                                    _stream(weight.device)))
    return out


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None,
           activation: Optional[str] = None, tensor_cores: bool = False,
           weight_split: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """F.linear (+ optional activation) on (..., K) rows.  tensor_cores=False: CUDA-core fp32 kernel
    (K % 16 == 0); True: tcgen05 kernel, TF32 hi·hi + one bf16 MMA for both corrections (K % 4 == 0, N % 4 == 0) — the one the model's
    token-sized projections run on; weight_split = split_tf32(weight) skips the per-call split; residual
    (same shape as the result, tensor_cores only) is added after the activation; out = preallocated result."""
    if x.device.type != "cuda":
        raise RuntimeError("linear runs on CUDA only (no CPU fallback)")
    x, weight, bias = map(_f32c, (x, weight, bias))
    K = x.shape[-1]
    N = weight.shape[0]
    x2 = x.reshape(-1, K)
    if out is None:
        out = torch.empty(x2.shape[0], N, device=x.device, dtype=torch.float32)
    if residual is not None:
        if not tensor_cores:
            raise NotImplementedError("residual is fused in the tensor-core kernel only")
        residual = _f32c(residual).reshape(-1, N)
    if x2.shape[0] > 0:
        lib = _native.lib()
        with torch.cuda.device(x.device):
            if tensor_cores:
                _native.check(lib.vasr_linear_tc(_native.ptr(x2), K, _native.ptr(weight), _native.ptr(weight_split),
                                                 _native.ptr(bias), _native.ptr(residual), N, _native.ptr(out), N,
                                                 x2.shape[0], K, N, _ACT[activation], _stream(x.device)))
            else:
                _native.check(lib.vasr_linear(_native.ptr(x2), K, _native.ptr(weight), _native.ptr(bias),
                                              _native.ptr(out), N, x2.shape[0], K, N, _ACT[activation],
                                              _stream(x.device)))
    return out.reshape(*x.shape[:-1], N)
