"""PointNet++ layer glue — the torch twin of the reference's utils/pointnet_util.py for the
set-abstraction / feature-propagation geometry path.

``sample_and_group`` / ``sample_and_group_all`` keep the reference's signatures and return tuples
(utils/pointnet_util.py:22-56, :59-84).  ``pointnet_sa_module``, ``pointnet_sa_module_msg`` and
``pointnet_fp_module`` keep the reference's full positional signatures (:87, :156, :199 — ``mlp`` lists of
widths, ``is_training``, ``bn_decay``, ``scope``, ``bn`` ...), so the reference's model files call them
unchanged; the dense half (1x1 conv + BN + ReLU stacks, :115-153, :187-195, :218-228) is cuDNN/cuBLAS
territory and outside this path: width lists resolve to torch layers kept in a variable-scope registry
(``layers.scoped_mlp``), or pass a callable, or None to get the grouped tensor pooled as-is.

``fused=True`` (default) routes through the fused kernels (FPS+gather in one launch,
group+centre+concat in one pass); ``fused=False`` issues the reference's exact op sequence.  Both
produce identical values.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence

import torch

from . import _lib, layers
from ._tensor import feature_dtype_code, on_device, ptr, require_cuda, same_device, stream_ptr
from .tf_grouping import group_point, knn_point, query_ball_point
from .tf_interpolate import fp_interpolate_concat, three_interpolate, three_nn, three_nn_interpolate
from .sa_layer import sample_group, sample_group_msg
from .tf_sampling import farthest_point_sample, farthest_point_sample_and_gather, gather_point


class _GroupConcat(torch.autograd.Function):
    """out = concat(xyz[idx]-new_xyz, points[idx]) in either channel order, plus grouped_xyz.  ``out`` has the dtype of
    ``points`` (float32 without points; the centred xyz rounded once into it), ``grouped_xyz`` is float32."""

    @staticmethod
    def forward(ctx, xyz, new_xyz, points, idx, xyz_first, dt):
        b, n, _ = xyz.shape
        _, m, s = idx.shape
        c = 0 if points is None else points.shape[2]
        dtype = torch.float32 if points is None else points.dtype
        out = torch.empty((b, m, s, 3 + c), dtype=dtype, device=xyz.device)
        gxyz = torch.empty((b, m, s, 3), dtype=torch.float32, device=xyz.device)
        if out.numel():
            lib = _lib.load()
            with on_device(xyz):
                args = (b, n, c, m, s, ptr(xyz), ptr(new_xyz), ptr(points), ptr(idx), 1 if xyz_first else 0, ptr(out),
                        ptr(gxyz), stream_ptr(xyz.device))
                rc = lib.pn2_group_concat_h(dt, *args) if dt else lib.pn2_group_concat(*args)
            _lib.check(rc, "pn2_group_concat")
        ctx.save_for_backward(idx)
        ctx.meta = (b, n, c, m, s, bool(xyz_first), points is not None, dt, dtype)
        return out, gxyz

    @staticmethod
    def backward(ctx, g_out, g_gxyz):
        (idx,) = ctx.saved_tensors
        b, n, c, m, s, xyz_first, has_points, dt, dtype = ctx.meta
        lib = _lib.load()
        dev = g_out.device
        lo = 0 if xyz_first else c
        g_xyz_part = g_out[..., lo:lo + 3]
        if dt:  # coordinates' gradient in float32, through the float32 kernel
            g_xyz_part = g_xyz_part.float()
        if g_gxyz is not None:
            g_xyz_part = g_xyz_part + g_gxyz
        g_xyz_part = g_xyz_part.contiguous()
        g_xyz = torch.zeros((b, n, 3), dtype=torch.float32, device=dev)
        g_points = None
        with on_device(g_out):
            st = stream_ptr(dev)
            _lib.check(lib.pn2_group_point_grad(b, n, 3, m, s, ptr(g_xyz_part), ptr(idx), ptr(g_xyz), st),
                       "pn2_group_point_grad")
            if has_points:
                g_feat = (g_out[..., 3:] if xyz_first else g_out[..., :c]).to(dtype).contiguous()
                g_points = torch.zeros((b, n, c), dtype=torch.float32, device=dev)
                if dt:  # 16-bit grad_out, accumulated in float32, rounded once
                    _lib.check(lib.pn2_group_point_grad_h(dt, b, n, c, m, s, ptr(g_feat), ptr(idx), ptr(g_points), st),
                               "pn2_group_point_grad_h")
                    g_points = g_points.to(dtype)
                else:
                    _lib.check(lib.pn2_group_point_grad(b, n, c, m, s, ptr(g_feat), ptr(idx), ptr(g_points), st),
                               "pn2_group_point_grad")
        g_new_xyz = -g_xyz_part.sum(dim=2)
        return g_xyz, g_new_xyz, g_points, None, None, None


def group_and_concat(xyz, new_xyz, points, idx, xyz_first: bool = True):
    """Fused tail of sample_and_group: returns (new_points (b,m,s,3+c), grouped_xyz (b,m,s,3)).

    ``points`` may be float32, bfloat16 or float16; new_points then has its dtype (features copied bit for bit, the
    centred xyz computed in float32 and rounded once).  xyz, new_xyz and grouped_xyz are float32."""
    dt = 0 if points is None else feature_dtype_code(points, "points")
    xyz = require_cuda(xyz, "xyz", torch.float32)
    new_xyz = require_cuda(new_xyz, "new_xyz", torch.float32)
    idx = require_cuda(idx, "idx", torch.int32)
    if points is not None:
        points = require_cuda(points, "points", points.dtype)
        same_device(xyz, new_xyz, idx, points)
        if points.dim() != 3 or points.shape[:2] != xyz.shape[:2]:
            raise ValueError("points must be (batch_size, ndataset, channel) matching xyz")
    else:
        same_device(xyz, new_xyz, idx)
    if idx.dim() != 3 or idx.shape[0] != xyz.shape[0] or new_xyz.shape[:2] != idx.shape[:2]:
        raise ValueError("idx must be (batch_size, npoint, nsample) matching new_xyz")
    return _GroupConcat.apply(xyz, new_xyz, points, idx, xyz_first, dt)


def sample_and_group(npoint, radius, nsample, xyz, points, knn=False, use_xyz=True, fused=True):
    """Sampling + grouping half of a set-abstraction layer (same positional arguments and return
    tuple as the reference's sample_and_group, utils/pointnet_util.py:22-56).

    Args:
        npoint, radius, nsample: centroids to sample, ball radius, neighbours kept per centroid.
        xyz (b, n, 3) float32; points (b, n, c) float32, bfloat16 or float16, or None (then the grouped xyz are
        the features).  new_points has the dtype of points; grouped_xyz is float32.
        knn: k-nearest-neighbour grouping instead of the ball query; use_xyz: keep the centred xyz
        in front of the grouped features.
    Returns:
        new_xyz (b, npoint, 3), new_points (b, npoint, nsample, 3 + c) [c alone when use_xyz is False],
        idx (b, npoint, nsample) int32 into the n input points, grouped_xyz (b, npoint, nsample, 3)
        centred on new_xyz.

    ``fused=True`` uses the overlapped sampling+grouping layer (sa_layer.sample_group) and the
    single-pass concat kernel; ``fused=False`` issues the reference's op sequence one by one.  Both
    return identical values.
    """
    no_grad_xyz = not xyz.requires_grad
    if fused and no_grad_xyz and not knn:
        # one call: FPS + gather + ball query (+ centred grouped xyz when they are the whole output)
        need_g = points is None or not use_xyz
        _, new_xyz, idx, _, grouped_xyz = sample_group(npoint, radius, nsample, xyz, center=True, want_grouped=need_g)
        if points is None:
            return new_xyz, grouped_xyz, idx, grouped_xyz
        if not use_xyz:
            return new_xyz, group_point(points, idx), idx, grouped_xyz
        new_points, grouped_xyz = group_and_concat(xyz, new_xyz, points, idx, xyz_first=True)
        return new_xyz, new_points, idx, grouped_xyz
    if fused and no_grad_xyz:
        _, new_xyz = farthest_point_sample_and_gather(npoint, xyz)
    else:
        new_xyz = gather_point(xyz, farthest_point_sample(npoint, xyz))
    if knn:
        _, idx = knn_point(nsample, xyz, new_xyz)
    else:
        idx, _ = query_ball_point(radius, nsample, xyz, new_xyz)
    if fused:
        feats = points if (points is not None and use_xyz) else None
        if points is not None and not use_xyz:
            grouped_xyz = group_point(xyz, idx) - new_xyz.unsqueeze(2)
            return new_xyz, group_point(points, idx), idx, grouped_xyz
        new_points, grouped_xyz = group_and_concat(xyz, new_xyz, feats, idx, xyz_first=True)
        return new_xyz, new_points, idx, grouped_xyz
    # the reference's sequence, op by op (:44-54)
    grouped_xyz = group_point(xyz, idx) - new_xyz.unsqueeze(2)
    if points is None:
        new_points = grouped_xyz
    else:
        grouped_points = group_point(points, idx)
        new_points = torch.cat([grouped_xyz, grouped_points], dim=-1) if use_xyz else grouped_points
    return new_xyz, new_points, idx, grouped_xyz


def sample_and_group_all(xyz, points, use_xyz=True):
    """The group_all variant (reference utils/pointnet_util.py:59-84): one group holding every point,
    centred on the origin — no sampling, no search, no kernel.

    Returns new_xyz (b, 1, 3) zeros, new_points (b, 1, n, 3 + c) (xyz first; c alone when use_xyz is
    False; the xyz themselves when points is None), idx (b, 1, n) = arange, grouped_xyz (b, 1, n, 3).
    """
    b, n = xyz.shape[0], xyz.shape[1]
    new_xyz = xyz.new_zeros((b, 1, 3))
    idx = torch.arange(n, dtype=torch.int32, device=xyz.device).view(1, 1, n).expand(b, 1, n).contiguous()
    grouped_xyz = xyz.view(b, 1, n, 3)
    if points is None:
        return new_xyz, grouped_xyz, idx, grouped_xyz
    new_points = (torch.cat([xyz, points], dim=2) if use_xyz else points).unsqueeze(1)
    return new_xyz, new_points, idx, grouped_xyz


def _apply_mlp(mlp, t: torch.Tensor, scope=None, name="mlp", bn=True, is_training=None, bn_decay=None) -> torch.Tensor:
    """``mlp`` is None (identity), a callable on a (..., channel) tensor, or — the reference's form — a list of
    output widths, resolved to the SharedMLP registered under ``scope/name`` (layers.scoped_mlp)."""
    if mlp is None:
        return t
    if callable(mlp):
        return mlp(t)
    widths = [int(w) for w in mlp]
    if not widths:
        return t
    return layers.scoped_mlp(scope, name, t.shape[-1], widths, bn, t.device, is_training, bn_decay)(t)


def pointnet_sa_module(xyz, points, npoint, radius, nsample, mlp=None, mlp2=None, group_all=False, is_training=None,
                       bn_decay=None, scope=None, bn=True, pooling='max', knn=False, use_xyz=True, use_nchw=False, fused=True):
    ''' PointNet Set Abstraction (SA) Module — same positional arguments as the reference
        (utils/pointnet_util.py:87-154), so its call sites run unchanged, e.g. models/pointnet2_sem_seg.py:28:
            pointnet_sa_module(l0_xyz, l0_points, npoint=1024, radius=0.1, nsample=32, mlp=[32,32,64], mlp2=None,
                               group_all=False, is_training=is_training, bn_decay=bn_decay, scope='layer1')
        mlp / mlp2: lists of output widths (layers live in the variable-scope registry, layers.scoped_mlp; is_training
        and bn_decay set their mode and batch-norm momentum), or callables on a (batch, npoint, nsample, channel) tensor,
        or None.  use_nchw is accepted and ignored (a layout hint for TensorFlow's conv2d).
        Return: new_xyz (b,npoint,3), new_points (b,npoint,channels), idx (b,npoint,nsample)
    '''
    if group_all:
        new_xyz, new_points, idx, grouped_xyz = sample_and_group_all(xyz, points, use_xyz)
    else:
        new_xyz, new_points, idx, grouped_xyz = sample_and_group(npoint, radius, nsample, xyz, points, knn, use_xyz,
                                                                 fused=fused)
    new_points = _apply_mlp(mlp, new_points, scope, "conv", bn, is_training, bn_decay)
    if pooling == 'max':
        new_points = new_points.max(dim=2, keepdim=True).values
    elif pooling == 'avg':
        new_points = new_points.mean(dim=2, keepdim=True)
    elif pooling == 'weighted_avg':
        dists = torch.linalg.vector_norm(grouped_xyz, ord=2, dim=-1, keepdim=True)
        exp_dists = torch.exp(-dists * 5)
        weights = exp_dists / exp_dists.sum(dim=2, keepdim=True)
        new_points = (new_points * weights).sum(dim=2, keepdim=True)
    elif pooling == 'max_and_avg':
        new_points = torch.cat([new_points.mean(dim=2, keepdim=True), new_points.max(dim=2, keepdim=True).values], dim=-1)
    else:
        raise ValueError(f"unknown pooling {pooling!r}")
    new_points = _apply_mlp(mlp2, new_points, scope, "conv_post", bn, is_training, bn_decay)
    return new_xyz, new_points.squeeze(2), idx


def pointnet_sa_module_msg(xyz, points, npoint, radius_list: Sequence[float], nsample_list: Sequence[int], mlp_list=None,
                           is_training=None, bn_decay=None, scope=None, bn=True, use_xyz=True, use_nchw=False, fused=True):
    ''' PointNet Set Abstraction (SA) module with Multi-Scale Grouping — same positional arguments as the
        reference (utils/pointnet_util.py:156-196).  One FPS+gather, then per scale: ball query, group,
        centre, concat in the MSG order [features, xyz] (:184), MLP, max-pool; scales concatenated.
        mlp_list: per scale a list of output widths (scope registry), a callable, or None.
        Return: new_xyz (b,npoint,3), new_points (b,npoint,sum of channels)
    '''
    pre = None
    if fused and not xyz.requires_grad and (points is None or use_xyz):
        # one call: the sampling pass and every scale's ball query (+ centred grouped xyz when they are the features)
        _, new_xyz, idx_list, _, gxyz_list = sample_group_msg(npoint, radius_list, nsample_list, xyz, center=True,
                                                              want_grouped=points is None)
        pre = (idx_list, gxyz_list)
    elif fused and not xyz.requires_grad:
        _, new_xyz = farthest_point_sample_and_gather(npoint, xyz)
    else:
        new_xyz = gather_point(xyz, farthest_point_sample(npoint, xyz))
    new_points_list = []
    for i in range(len(radius_list)):
        radius, nsample = radius_list[i], nsample_list[i]
        if pre is not None:
            idx = pre[0][i]
            if points is None:
                grouped_points = pre[1][i]
            else:
                grouped_points, _ = group_and_concat(xyz, new_xyz, points, idx, xyz_first=False)
        else:
            idx, pts_cnt = query_ball_point(radius, nsample, xyz, new_xyz)
            if fused and (points is None or use_xyz):
                grouped_points, _ = group_and_concat(xyz, new_xyz, points, idx, xyz_first=False)
            else:
                grouped_xyz = group_point(xyz, idx) - new_xyz.unsqueeze(2)
                if points is not None:
                    grouped_points = group_point(points, idx)
                    if use_xyz:
                        grouped_points = torch.cat([grouped_points, grouped_xyz], dim=-1)
                else:
                    grouped_points = grouped_xyz
        grouped_points = _apply_mlp(None if mlp_list is None else mlp_list[i], grouped_points, scope, f"conv{i}", bn, is_training, bn_decay)
        new_points_list.append(grouped_points.max(dim=2).values)
    return new_xyz, torch.cat(new_points_list, dim=-1)


def pointnet_fp_module(xyz1, xyz2, points1, points2, mlp=None, is_training=None, bn_decay=None, scope=None, bn=True, fused=True):
    ''' PointNet Feature Propogation (FP) Module — same positional arguments as the reference
        (utils/pointnet_util.py:199-229).
        xyz1 (b,n1,3) dense, xyz2 (b,n2,3) sparser, points1 (b,n1,c1) or None, points2 (b,n2,c2);
        mlp: list of output widths (scope registry), a callable on a (b,n1,1,channel) tensor, or None.
        Return: new_points (b,n1,mlp[-1]) (or (b,n1,c2+c1) when mlp is None)
    '''
    no_grad = not points2.requires_grad and (points1 is None or not points1.requires_grad)
    # the fused kernel takes one feature dtype; mixed ones go through torch.cat, which promotes
    one_dtype = points1 is None or points1.dtype == points2.dtype
    if fused and no_grad and one_dtype and points2.shape[2] > 0:
        # one kernel: 3-NN, weights, interpolation and the concat of :219
        new_points1 = fp_interpolate_concat(xyz1, xyz2, points1, points2)
    else:
        if fused and not points2.requires_grad:
            interpolated_points = three_nn_interpolate(xyz1, xyz2, points2)
        else:
            dist, idx = three_nn(xyz1, xyz2)
            dist = torch.clamp(dist, min=1e-10)
            norm = (1.0 / dist).sum(dim=2, keepdim=True)
            weight = (1.0 / dist) / norm
            interpolated_points = three_interpolate(points2, idx, weight)
        if points1 is not None:
            new_points1 = torch.cat([interpolated_points, points1], dim=2)  # B,ndataset1,nchannel1+nchannel2
        else:
            new_points1 = interpolated_points
    if mlp is not None:
        new_points1 = _apply_mlp(mlp, new_points1.unsqueeze(2), scope, "conv", bn, is_training, bn_decay).squeeze(2)
    return new_points1
