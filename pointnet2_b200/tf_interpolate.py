"""Interpolation ops — drop-in for the reference's tf_ops/3d_interpolation/tf_interpolate.py.

Same names, argument order and returns as tf_interpolate.py:8-34, on contiguous CUDA torch
tensors.  The reference only has CPU kernels for these (tf_interpolate.cpp:187,222,262), so
TensorFlow bounces the tensors through host memory; here they run on the device.
three_interpolate is differentiable w.r.t. ``points`` only (tf_interpolate.py:29-34); three_nn has
no gradient (:18).
"""
from __future__ import annotations

import torch

from . import _lib
from ._tensor import feature_dtype_code, on_device, ptr, require_cuda, same_device, stream_ptr


def three_nn(xyz1: torch.Tensor, xyz2: torch.Tensor):
    """The three nearest known points of every unknown point.

    ``xyz1`` float32 (B, n, 3): the points that need values; ``xyz2`` float32 (B, m, 3): the points that carry them.
    Returns ``dist`` float32 (B, n, 3) — SQUARED distances, ascending — and ``idx`` int32 (B, n, 3), positions in
    ``xyz2``.
    Reference: tf_interpolate.py:8-17 -> ThreeNNOp (tf_interpolate.cpp:157-187) -> threenn_cpu (:60-103).
    """
    xyz1 = require_cuda(xyz1, "xyz1", torch.float32)
    xyz2 = require_cuda(xyz2, "xyz2", torch.float32)
    same_device(xyz1, xyz2)
    if xyz1.dim() != 3 or xyz1.shape[2] != 3:
        raise ValueError(f"ThreeNN expects (b,n,3) xyz1 shape, got {tuple(xyz1.shape)}")
    if xyz2.dim() != 3 or xyz2.shape[2] != 3 or xyz2.shape[0] != xyz1.shape[0]:
        raise ValueError(f"ThreeNN expects (b,m,3) xyz2 shape, got {tuple(xyz2.shape)}")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    dist = torch.empty((b, n, 3), dtype=torch.float32, device=xyz1.device)
    idx = torch.empty((b, n, 3), dtype=torch.int32, device=xyz1.device)
    if b * n:
        with on_device(xyz1):
            rc = _lib.load().pn2_three_nn(b, n, m, ptr(xyz1), ptr(xyz2), ptr(dist), ptr(idx), stream_ptr(xyz1.device))
        _lib.check(rc, "pn2_three_nn")
    return dist, idx


# three_interpolate's backward: True = inverse index + ordered sums (run-to-run deterministic, bit-identical to the
# reference's CPU function on non-degenerate layers); False = the float-atomic scatter (the reference-signature
# pn2_three_interpolate_grad, the reference's own semantics on a GPU).  Measured at 16 x 8192 <- 1024, C = 128
# (profiles/r2_report.json): see DESIGN.md section 5.4 for which is faster where.
DETERMINISTIC_GRAD = True


class _ThreeInterpolate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, idx, weight, dt):
        b, m, c = points.shape
        n = idx.shape[1]
        out = torch.empty((b, n, c), dtype=points.dtype, device=points.device)
        if out.numel():
            lib = _lib.load()
            with on_device(points):
                if dt:
                    rc = lib.pn2_three_interpolate_h(dt, b, m, c, n, ptr(points), ptr(idx), ptr(weight), ptr(out),
                                                     stream_ptr(points.device))
                else:
                    rc = lib.pn2_three_interpolate(b, m, c, n, ptr(points), ptr(idx), ptr(weight), ptr(out),
                                                   stream_ptr(points.device))
            _lib.check(rc, "pn2_three_interpolate")
        ctx.save_for_backward(idx, weight)
        ctx.shape = (b, m, c)
        ctx.dt = (dt, points.dtype)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        idx, weight = ctx.saved_tensors
        b, m, c = ctx.shape
        n = idx.shape[1]
        dt, dtype = ctx.dt
        grad_out = grad_out.to(dtype).contiguous()
        lib = _lib.load()
        dev = grad_out.device
        # 16-bit gradients: the _h entries read the 16-bit grad_out and accumulate in float32, rounded once here
        if DETERMINISTIC_GRAD and b * m * c:
            # inverse index + ordered accumulation: deterministic, bit-identical to threeinterpolate_grad_cpu
            # (tf_interpolate.cpp:131-153), and ~3x faster than the atomics at the sem-seg sizes
            grad_points = torch.empty((b, m, c), dtype=torch.float32, device=dev)
            with on_device(grad_out):
                wsb = int(lib.pn2_three_interpolate_grad_det_workspace_bytes(b, max(n, 1), m))
                ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
                if dt:
                    rc = lib.pn2_three_interpolate_grad_det_h(dt, b, n, c, m, ptr(grad_out), ptr(idx), ptr(weight),
                                                              ptr(grad_points), ptr(ws), wsb, stream_ptr(dev))
                else:
                    rc = lib.pn2_three_interpolate_grad_det(b, n, c, m, ptr(grad_out), ptr(idx), ptr(weight), ptr(grad_points),
                                                            ptr(ws), wsb, stream_ptr(dev))
            _lib.check(rc, "pn2_three_interpolate_grad_det")
            return grad_points.to(dtype), None, None, None
        # zero-filled by the caller, as ThreeInterpolateGradOp does (tf_interpolate.cpp:258)
        grad_points = torch.zeros((b, m, c), dtype=torch.float32, device=dev)
        if grad_out.numel():
            with on_device(grad_out):
                if dt:
                    rc = lib.pn2_three_interpolate_grad_h(dt, b, n, c, m, ptr(grad_out), ptr(idx), ptr(weight),
                                                          ptr(grad_points), stream_ptr(dev))
                else:
                    rc = lib.pn2_three_interpolate_grad(b, n, c, m, ptr(grad_out), ptr(idx), ptr(weight),
                                                        ptr(grad_points), stream_ptr(dev))
            _lib.check(rc, "pn2_three_interpolate_grad")
        return grad_points.to(dtype), None, None, None


def three_interpolate(points: torch.Tensor, idx: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """Weighted sum of three feature rows: ``out[b, i, :] = sum_t weight[b, i, t] * points[b, idx[b, i, t], :]``.

    ``points`` float32, bfloat16 or float16 (B, m, c): features of the known points; ``idx`` int32 and ``weight``
    float32, both (B, n, 3), as produced from three_nn.  Returns (B, n, c) of the dtype of ``points``: 16-bit features
    are widened exactly, interpolated in float32 and rounded once.  Differentiable in ``points``.
    Reference: tf_interpolate.py:19-28 -> threeinterpolate_cpu (tf_interpolate.cpp:107-127);
    gradient :29-34 -> threeinterpolate_grad_cpu (:131-153).
    """
    dt = feature_dtype_code(points, "points")
    points = require_cuda(points, "points", points.dtype)
    idx = require_cuda(idx, "idx", torch.int32)
    weight = require_cuda(weight, "weight", torch.float32)
    same_device(points, idx, weight)
    if points.dim() != 3:
        raise ValueError(f"ThreeInterpolate expects (b,m,c) points shape, got {tuple(points.shape)}")
    b = points.shape[0]
    if idx.dim() != 3 or idx.shape[0] != b or idx.shape[2] != 3:
        raise ValueError(f"ThreeInterpolate expects (b,n,3) idx shape, got {tuple(idx.shape)}")
    if weight.dim() != 3 or tuple(weight.shape) != tuple(idx.shape):
        raise ValueError(f"ThreeInterpolate expects (b,n,3) weight shape, got {tuple(weight.shape)}")
    if points.shape[1] <= 0 and idx.numel():
        raise ValueError("ThreeInterpolate expects a non-empty points tensor")
    return _ThreeInterpolate.apply(points, idx, weight.detach(), dt)


def three_nn_interpolate(xyz1: torch.Tensor, xyz2: torch.Tensor, points2: torch.Tensor, return_aux: bool = False):
    """Fused feature-propagation front end (utils/pointnet_util.py:211-216): three_nn, the
    inverse-distance weights (dist=max(dist,1e-10); w=(1/dist)/sum(1/dist)) and three_interpolate
    in one kernel; dist/idx/weight stay on chip unless ``return_aux``.  Forward only (use the
    unfused ops when ``points2`` needs a gradient).  ``points2`` may be float32, bfloat16 or float16; ``out`` has its
    dtype (interpolated in float32, rounded once), dist / weight are float32.
    Returns out (b,n,c) [, dist (b,n,3), idx (b,n,3), weight (b,n,3)]."""
    dt = feature_dtype_code(points2, "points2")
    xyz1 = require_cuda(xyz1, "xyz1", torch.float32)
    xyz2 = require_cuda(xyz2, "xyz2", torch.float32)
    points2 = require_cuda(points2, "points2", points2.dtype)
    same_device(xyz1, xyz2, points2)
    if xyz1.dim() != 3 or xyz1.shape[2] != 3 or xyz2.dim() != 3 or xyz2.shape[2] != 3 or xyz1.shape[0] != xyz2.shape[0]:
        raise ValueError("three_nn_interpolate expects (b,n,3) xyz1 and (b,m,3) xyz2")
    if points2.dim() != 3 or points2.shape[:2] != xyz2.shape[:2]:
        raise ValueError("three_nn_interpolate expects (b,m,c) points2 matching xyz2")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    c = points2.shape[2]
    if m <= 0:
        raise ValueError("three_nn_interpolate expects at least one known point")
    dev = xyz1.device
    out = torch.empty((b, n, c), dtype=points2.dtype, device=dev)
    dist = torch.empty((b, n, 3), dtype=torch.float32, device=dev) if return_aux else None
    idx = torch.empty((b, n, 3), dtype=torch.int32, device=dev) if return_aux else None
    weight = torch.empty((b, n, 3), dtype=torch.float32, device=dev) if return_aux else None
    if b * n:
        lib = _lib.load()
        with on_device(xyz1):
            args = (b, n, m, c, ptr(xyz1), ptr(xyz2), ptr(points2.detach()), ptr(out), ptr(dist), ptr(idx), ptr(weight),
                    stream_ptr(dev))
            rc = lib.pn2_three_nn_interpolate_h(dt, *args) if dt else lib.pn2_three_nn_interpolate(*args)
        _lib.check(rc, "pn2_three_nn_interpolate")
    if return_aux:
        return out, dist, idx, weight
    return out


def fp_interpolate_concat(xyz1: torch.Tensor, xyz2: torch.Tensor, points1, points2: torch.Tensor) -> torch.Tensor:
    """The front end of pointnet_fp_module in one kernel (utils/pointnet_util.py:211-219): three_nn, the
    inverse-distance weights, three_interpolate AND the concat with ``points1``:
    returns (b, n, c2 + c1) = [interpolated points2 | points1] (c1 = 0 when ``points1`` is None).  Forward only.
    ``points1`` and ``points2`` are float32, bfloat16 or float16, both of the same dtype, which the output has."""
    dt = feature_dtype_code(points2, "points2")
    if points1 is not None:
        feature_dtype_code(points1, "points1")
        if points1.dtype != points2.dtype:
            raise TypeError(f"fp_interpolate_concat expects points1 and points2 of one dtype, got {points1.dtype} and {points2.dtype}")
    xyz1 = require_cuda(xyz1, "xyz1", torch.float32)
    xyz2 = require_cuda(xyz2, "xyz2", torch.float32)
    points2 = require_cuda(points2, "points2", points2.dtype)
    same_device(xyz1, xyz2, points2)
    if xyz1.dim() != 3 or xyz1.shape[2] != 3 or xyz2.dim() != 3 or xyz2.shape[2] != 3 or xyz1.shape[0] != xyz2.shape[0]:
        raise ValueError("fp_interpolate_concat expects (b,n,3) xyz1 and (b,m,3) xyz2")
    if points2.dim() != 3 or points2.shape[:2] != xyz2.shape[:2]:
        raise ValueError("fp_interpolate_concat expects (b,m,c2) points2 matching xyz2")
    b, n, _ = xyz1.shape
    m, c2 = xyz2.shape[1], points2.shape[2]
    c1 = 0
    if points1 is not None:
        points1 = require_cuda(points1, "points1", points1.dtype)
        same_device(xyz1, points1)
        if points1.dim() != 3 or points1.shape[:2] != xyz1.shape[:2]:
            raise ValueError("fp_interpolate_concat expects (b,n,c1) points1 matching xyz1")
        c1 = points1.shape[2]
    if m <= 0 or c2 <= 0:
        raise ValueError("fp_interpolate_concat expects at least one known point and one channel")
    out = torch.empty((b, n, c2 + c1), dtype=points2.dtype, device=xyz1.device)
    if b * n:
        lib = _lib.load()
        with on_device(xyz1):
            args = (b, n, m, c2, c1, ptr(xyz1), ptr(xyz2), ptr(points1.detach()) if c1 else None, ptr(points2.detach()),
                    ptr(out), stream_ptr(xyz1.device))
            rc = lib.pn2_fp_interpolate_concat_h(dt, *args) if dt else lib.pn2_fp_interpolate_concat(*args)
        _lib.check(rc, "pn2_fp_interpolate_concat")
    return out
