"""Argument checking shared by the op wrappers.

Mirrors the reference OpKernels' OP_REQUIRES checks (tf_ops/sampling/tf_sampling.cpp:99,105,131,135;
tf_ops/grouping/tf_grouping.cpp:71-84,90,96; tf_ops/3d_interpolation/tf_interpolate.cpp:163-168,
197-206): shape / attribute violations raise ValueError (TensorFlow: InvalidArgument), wrong dtypes
raise TypeError.  Tensors must live on a CUDA device: there is no CPU path.
"""
from __future__ import annotations

import ctypes
from contextlib import contextmanager

import torch


def require_cuda(t: torch.Tensor, name: str, dtype: torch.dtype) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: pointnet2_b200 has no CPU path "
                           f"(got device {t.device})")
    return t if t.is_contiguous() else t.contiguous()


# feature dtypes and their codes in the C ABI (include/pn2_api.h: PN2_DTYPE_BF16, PN2_DTYPE_F16; 0 = float32, which
# calls the float32 entry points)
FEATURE_DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def feature_dtype_code(t, name: str) -> int:
    """Features may be float32, bfloat16 or float16 (coordinates and weights stay float32): the ABI dtype code of
    ``t``, TypeError for anything else."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    code = FEATURE_DTYPES.get(t.dtype)
    if code is None:
        raise TypeError(f"{name} must be torch.float32, torch.bfloat16 or torch.float16, got {t.dtype}")
    return code


def same_device(*ts: torch.Tensor) -> None:
    dev = ts[0].device
    for t in ts[1:]:
        if t.device != dev:
            raise RuntimeError(f"all tensors must be on the same device ({dev} vs {t.device})")


def ptr(t) -> ctypes.c_void_p:
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


@contextmanager
def on_device(t: torch.Tensor):
    with torch.cuda.device(t.device):
        yield
