"""Grouping ops — drop-in for the reference's tf_ops/grouping/tf_grouping.py.

Same function names, positional order and return tuples as tf_grouping.py:8-73 on contiguous CUDA
torch tensors.  group_point is differentiable w.r.t. ``points`` (tf_grouping.py:42-46);
query_ball_point / select_top_k have no gradient (ops.NoGradient, :21,:32).
"""
from __future__ import annotations

import torch

from . import _lib
from ._tensor import feature_dtype_code, on_device, ptr, require_cuda, same_device, stream_ptr


def query_ball_point(radius: float, nsample: int, xyz1: torch.Tensor, xyz2: torch.Tensor):
    """For every query centre, the first ``nsample`` data points (ascending index) closer than ``radius``.

    Arguments: ``radius`` of the ball; ``nsample`` row length; ``xyz1`` float32 (B, N, 3), the cloud that is
    searched; ``xyz2`` float32 (B, M, 3), the ball centres.
    Returns ``idx`` int32 (B, M, nsample) — positions in ``xyz1``, short rows padded with their first hit — and
    ``pts_cnt`` int32 (B, M), how many distinct hits each row holds.
    Reference: tf_grouping.py:8-20 -> QueryBallPointGpuOp (tf_grouping.cpp:67-106) ->
    query_ball_point_gpu (tf_grouping_g.cu:3-36).  Rows with no point in the ball (undefined in the
    reference) come back as zeros with pts_cnt 0.
    """
    radius = float(radius)
    nsample = int(nsample)
    if not radius > 0:
        raise ValueError("QueryBallPoint expects positive radius")
    if nsample <= 0:
        raise ValueError("QueryBallPoint expects positive nsample")
    xyz1 = require_cuda(xyz1, "xyz1", torch.float32)
    xyz2 = require_cuda(xyz2, "xyz2", torch.float32)
    same_device(xyz1, xyz2)
    if xyz1.dim() != 3 or xyz1.shape[2] != 3:
        raise ValueError(f"QueryBallPoint expects (batch_size, ndataset, 3) xyz1 shape, got {tuple(xyz1.shape)}")
    if xyz2.dim() != 3 or xyz2.shape[2] != 3 or xyz2.shape[0] != xyz1.shape[0]:
        raise ValueError(f"QueryBallPoint expects (batch_size, npoint, 3) xyz2 shape, got {tuple(xyz2.shape)}")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    if n <= 0 and b * m:
        raise ValueError("QueryBallPoint expects a non-empty xyz1")
    idx = torch.empty((b, m, nsample), dtype=torch.int32, device=xyz1.device)
    pts_cnt = torch.empty((b, m), dtype=torch.int32, device=xyz1.device)
    if b * m:
        lib = _lib.load()
        with on_device(xyz1):
            ws_bytes = int(lib.pn2_query_ball_point_workspace_bytes(b, n))
            if ws_bytes:  # sparse balls are served through a uniform grid built in this scratch
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=xyz1.device)
                rc = lib.pn2_query_ball_point_ws(b, n, m, radius, nsample, ptr(xyz1), ptr(xyz2), ptr(idx), ptr(pts_cnt),
                                                 ptr(ws), ws_bytes, stream_ptr(xyz1.device))
            else:
                rc = lib.pn2_query_ball_point(b, n, m, radius, nsample, ptr(xyz1), ptr(xyz2), ptr(idx),
                                              ptr(pts_cnt), stream_ptr(xyz1.device))
        _lib.check(rc, "pn2_query_ball_point")
    return idx, pts_cnt


def select_top_k(k: int, dist: torch.Tensor):
    """k rounds of selection sort along the last axis of a distance matrix.

    Arguments: ``k`` — how many of the smallest entries to bring to the front; ``dist`` float32 (B, M, N), one row
    of N distances per query.
    Returns ``(idx, dist_out)``, both (B, M, N): columns [0, k) hold the k smallest distances in ascending order and
    their original column numbers, the remaining columns the reference's swapped-around tail.
    Reference: tf_grouping.py:22-31 -> SelectionSortGpuOp (tf_grouping.cpp:110-139) ->
    selection_sort_gpu (tf_grouping_g.cu:83-123).
    """
    k = int(k)
    if k <= 0:
        raise ValueError("SelectionSort expects positive k")
    dist = require_cuda(dist, "dist", torch.float32)
    if dist.dim() != 3:
        raise ValueError(f"SelectionSort expects (b,m,n) dist shape, got {tuple(dist.shape)}")
    b, m, n = dist.shape
    outi = torch.empty((b, m, n), dtype=torch.int32, device=dist.device)
    out = torch.empty((b, m, n), dtype=torch.float32, device=dist.device)
    if b * m * n:
        with on_device(dist):
            rc = _lib.load().pn2_selection_sort(b, n, m, k, ptr(dist), ptr(outi), ptr(out), stream_ptr(dist.device))
        _lib.check(rc, "pn2_selection_sort")
    return outi, out


class _GroupPoint(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, idx, dt):
        b, n, c = points.shape
        _, m, s = idx.shape
        out = torch.empty((b, m, s, c), dtype=points.dtype, device=points.device)
        if out.numel():
            lib = _lib.load()
            with on_device(points):
                if dt:
                    rc = lib.pn2_group_point_h(dt, b, n, c, m, s, ptr(points), ptr(idx), ptr(out), stream_ptr(points.device))
                else:
                    rc = lib.pn2_group_point(b, n, c, m, s, ptr(points), ptr(idx), ptr(out), stream_ptr(points.device))
            _lib.check(rc, "pn2_group_point")
        ctx.save_for_backward(idx)
        ctx.shape = (b, n, c)
        ctx.dt = (dt, points.dtype)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (idx,) = ctx.saved_tensors
        b, n, c = ctx.shape
        _, m, s = idx.shape
        dt, dtype = ctx.dt
        grad_out = grad_out.to(dtype).contiguous()
        # zero-filled by the caller, as GroupPointGradGpuOp does (tf_grouping.cpp:204); 16-bit gradients accumulate in
        # float32 and are rounded once
        grad_points = torch.zeros((b, n, c), dtype=torch.float32, device=grad_out.device)
        if grad_out.numel():
            lib = _lib.load()
            with on_device(grad_out):
                if dt:
                    rc = lib.pn2_group_point_grad_h(dt, b, n, c, m, s, ptr(grad_out), ptr(idx), ptr(grad_points),
                                                    stream_ptr(grad_out.device))
                else:
                    rc = lib.pn2_group_point_grad(b, n, c, m, s, ptr(grad_out), ptr(idx), ptr(grad_points),
                                                  stream_ptr(grad_out.device))
            _lib.check(rc, "pn2_group_point_grad")
        return grad_points.to(dtype), None, None


def group_point(points: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """Row gather: ``out[b, j, s, :] = points[b, idx[b, j, s], :]``.

    Arguments: ``points`` float32, bfloat16 or float16 (B, N, C), the rows to pick from; ``idx`` int32 (B, M, S), row
    numbers into ``points``.  Returns (B, M, S, C) of the dtype of ``points``, bit for bit.  Differentiable in
    ``points``; a 16-bit gradient is accumulated in float32 and rounded once.
    Reference: tf_grouping.py:33-41 -> group_point_gpu (tf_grouping_g.cu:40-57); gradient
    tf_grouping.py:42-46 -> group_point_grad_gpu (:61-78).
    """
    dt = feature_dtype_code(points, "points")
    points = require_cuda(points, "points", points.dtype)
    idx = require_cuda(idx, "idx", torch.int32)
    same_device(points, idx)
    if points.dim() != 3:
        raise ValueError(f"GroupPoint expects (batch_size, num_points, channel) points shape, got {tuple(points.shape)}")
    if idx.dim() != 3 or idx.shape[0] != points.shape[0]:
        raise ValueError(f"GroupPoint expects (batch_size, npoints, nsample) idx shape, got {tuple(idx.shape)}")
    if points.shape[1] <= 0 and idx.numel():
        raise ValueError("GroupPoint expects a non-empty points tensor")
    return _GroupPoint.apply(points, idx, dt)


def knn_point(k: int, xyz1: torch.Tensor, xyz2: torch.Tensor):
    """The k nearest data points of every query point, by squared Euclidean distance.

    Arguments: ``k`` neighbours per query; ``xyz1`` float32 (B, N, c), the cloud that is searched; ``xyz2`` float32
    (B, M, c), the queries.  Returns ``val`` float32 (B, M, k), the squared distances in ascending order, and
    ``idx`` int32 (B, M, k), the matching positions in ``xyz1``.
    Reference: tf_grouping.py:48-73.  The reference builds the (b,m,n) matrix of squared distances
    sum((xyz1 - xyz2)**2, -1) and runs select_top_k on it; for 3-D points and k <= 128 this runs one
    tiled top-k kernel instead (pn2_knn_point: no matrix), whose val / idx equal the first k columns
    of that composite bit for bit, ties included.  Other shapes take the composite itself.
    """
    k = int(k)
    if k <= 0:
        raise ValueError("knn_point expects positive k")
    xyz1 = require_cuda(xyz1, "xyz1", torch.float32)
    xyz2 = require_cuda(xyz2, "xyz2", torch.float32)
    same_device(xyz1, xyz2)
    if xyz1.dim() != 3 or xyz2.dim() != 3 or xyz1.shape[0] != xyz2.shape[0] or xyz1.shape[2] != xyz2.shape[2]:
        raise ValueError("knn_point expects (b,n,c) xyz1 and (b,m,c) xyz2")
    b, n, c = xyz1.shape
    m = xyz2.shape[1]
    if k > n:
        raise ValueError(f"knn_point expects k <= ndataset (the reference slices k columns of an n-column matrix), got k={k}, n={n}")
    if c == 3 and k <= 128:
        val = torch.empty((b, m, k), dtype=torch.float32, device=xyz1.device)
        idx = torch.empty((b, m, k), dtype=torch.int32, device=xyz1.device)
        if b * m:
            with on_device(xyz1):
                rc = _lib.load().pn2_knn_point(b, n, m, k, ptr(xyz1.detach()), ptr(xyz2.detach()), ptr(val), ptr(idx),
                                               stream_ptr(xyz1.device))
            _lib.check(rc, "pn2_knn_point")
        return val, idx
    diff = xyz1.unsqueeze(1) - xyz2.unsqueeze(2)  # (b,m,n,c): tile(xyz1) - tile(xyz2), tf_grouping.py:64-66
    dist = (diff * diff).sum(-1)
    outi, out = select_top_k(k, dist)
    return out[:, :, :k].contiguous(), outi[:, :, :k].contiguous()
