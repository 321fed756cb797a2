"""ctypes front-end of the oracle — TEST INFRASTRUCTURE ONLY (see oracle/pn2_oracle.c header).

Three families, all taking/returning numpy arrays unless noted:

* ``oracle_*``   — the C restatement (oracle/liboracle.so).
* ``refcpu_*``   — the reference's own CPU functions built from /root/reference
                   (oracle/_ref/libref_cpu.so): query_ball_point_cpu, group_point_cpu(+grad),
                   threenn_cpu, threeinterpolate_cpu(+grad), selection_sort_cpu.
* ``refcuda_*``  — the reference's own CUDA launchers rebuilt for sm_100a
                   (oracle/_ref/libref_{sampling,grouping}.so); these take CUDA torch tensors and
                   launch on the legacy default stream exactly as the reference does
                   (tf_sampling_g.cu:203-211, tf_grouping_g.cu:125-141).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_F = np.float32
_I = np.int32


def _build():
    import importlib.util
    spec = importlib.util.spec_from_file_location("pn2_oracle_build", os.path.join(HERE, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_lib = None
_refcpu = None
_refcuda = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        path = os.path.join(HERE, "liboracle.so")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(os.path.join(HERE, "pn2_oracle.c")):
            path = _build().build_oracle()
        _lib = ctypes.CDLL(path)
        _lib.oracle_ball_threshold.restype = c_float
        _lib.oracle_ball_threshold.argtypes = [c_float]
    return _lib


def have_refcpu() -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", "libref_cpu.so"))


def have_refcuda() -> bool:
    d = os.path.join(HERE, "_ref")
    return all(os.path.exists(os.path.join(d, n)) for n in ("libref_sampling.so", "libref_grouping.so"))


def refcpu() -> ctypes.CDLL:
    global _refcpu
    if _refcpu is None:
        path = os.path.join(HERE, "_ref", "libref_cpu.so")
        if not os.path.exists(path):
            _build().build_ref()
        _refcpu = ctypes.CDLL(path)
    return _refcpu


def refcuda():
    global _refcuda
    if _refcuda is None:
        d = os.path.join(HERE, "_ref")
        if not have_refcuda():
            _build().build_ref()
        _refcuda = (ctypes.CDLL(os.path.join(d, "libref_sampling.so")),
                    ctypes.CDLL(os.path.join(d, "libref_grouping.so")))
    return _refcuda


def _f(a):
    return np.ascontiguousarray(a, dtype=_F)


def _i(a):
    return np.ascontiguousarray(a, dtype=_I)


def _p(a):
    return a.ctypes.data_as(c_void_p)


# ----------------------------------------------------------------------------- C restatement
def oracle_fps(npoint: int, xyz, keyorder: bool = False):
    xyz = _f(xyz)
    b, n, _ = xyz.shape
    out = np.zeros((b, npoint), _I)
    fn = lib().oracle_fps_keyorder if keyorder else lib().oracle_fps
    fn(c_int(b), c_int(n), c_int(npoint), _p(xyz), _p(out))
    return out


def oracle_prob_cumsum(inp):
    inp = _f(inp)
    b, n = inp.shape
    out = np.empty((b, n), _F)
    lib().oracle_prob_cumsum(c_int(b), c_int(n), _p(inp), _p(out))
    return out


def oracle_prob_sample(inp, inpr):
    inp, inpr = _f(inp), _f(inpr)
    b, n = inp.shape
    m = inpr.shape[1]
    temp = np.empty((b, n), _F)
    out = np.empty((b, m), _I)
    lib().oracle_prob_sample(c_int(b), c_int(n), c_int(m), _p(inp), _p(inpr), _p(temp), _p(out))
    return out


def oracle_gather_point(inp, idx):
    inp, idx = _f(inp), _i(idx)
    b, n, _ = inp.shape
    m = idx.shape[1]
    out = np.empty((b, m, 3), _F)
    lib().oracle_gather_point(c_int(b), c_int(n), c_int(m), _p(inp), _p(idx), _p(out))
    return out


def oracle_gather_point_grad(inp_shape, idx, out_g):
    idx, out_g = _i(idx), _f(out_g)
    b, n, _ = inp_shape
    m = idx.shape[1]
    g = np.zeros((b, n, 3), _F)
    lib().oracle_gather_point_grad(c_int(b), c_int(n), c_int(m), _p(out_g), _p(idx), _p(g))
    return g


def oracle_query_ball_point(radius: float, nsample: int, xyz1, xyz2, use_fma: bool = True):
    xyz1, xyz2 = _f(xyz1), _f(xyz2)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    idx = np.zeros((b, m, nsample), _I)
    cnt = np.zeros((b, m), _I)
    lib().oracle_query_ball_point(c_int(b), c_int(n), c_int(m), c_float(radius), c_int(nsample),
                                  _p(xyz1), _p(xyz2), _p(idx), _p(cnt), c_int(1 if use_fma else 0))
    return idx, cnt


def oracle_ball_threshold(radius: float) -> float:
    return float(lib().oracle_ball_threshold(c_float(radius)))


def oracle_group_point(points, idx):
    points, idx = _f(points), _i(idx)
    b, n, c = points.shape
    _, m, s = idx.shape
    out = np.empty((b, m, s, c), _F)
    lib().oracle_group_point(c_int(b), c_int(n), c_int(c), c_int(m), c_int(s), _p(points), _p(idx), _p(out))
    return out


def oracle_group_point_grad(points_shape, idx, grad_out):
    idx, grad_out = _i(idx), _f(grad_out)
    b, n, c = points_shape
    _, m, s = idx.shape
    g = np.zeros((b, n, c), _F)
    lib().oracle_group_point_grad(c_int(b), c_int(n), c_int(c), c_int(m), c_int(s), _p(grad_out), _p(idx), _p(g))
    return g


def oracle_three_nn(xyz1, xyz2):
    xyz1, xyz2 = _f(xyz1), _f(xyz2)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    dist = np.empty((b, n, 3), _F)
    idx = np.empty((b, n, 3), _I)
    lib().oracle_three_nn(c_int(b), c_int(n), c_int(m), _p(xyz1), _p(xyz2), _p(dist), _p(idx))
    return dist, idx


def oracle_three_interpolate(points, idx, weight):
    points, idx, weight = _f(points), _i(idx), _f(weight)
    b, m, c = points.shape
    n = idx.shape[1]
    out = np.empty((b, n, c), _F)
    lib().oracle_three_interpolate(c_int(b), c_int(m), c_int(c), c_int(n), _p(points), _p(idx), _p(weight), _p(out))
    return out


def oracle_three_interpolate_grad(points_shape, idx, weight, grad_out):
    idx, weight, grad_out = _i(idx), _f(weight), _f(grad_out)
    b, m, c = points_shape
    n = idx.shape[1]
    g = np.zeros((b, m, c), _F)
    lib().oracle_three_interpolate_grad(c_int(b), c_int(n), c_int(c), c_int(m), _p(grad_out), _p(idx), _p(weight), _p(g))
    return g


def oracle_selection_sort(k: int, dist):
    dist = _f(dist)
    b, m, n = dist.shape
    outi = np.empty((b, m, n), _I)
    out = np.empty((b, m, n), _F)
    lib().oracle_selection_sort(c_int(b), c_int(n), c_int(m), c_int(k), _p(dist), _p(outi), _p(out))
    return outi, out


def oracle_knn_point(k: int, xyz1, xyz2):
    """knn_point as the reference composes it (tf_grouping.py:48-73): the (b,m,n) matrix of squared distances
    sum((xyz1 - xyz2)**2, -1) — element-wise float32 squares summed left to right — then selection sort
    (oracle_selection_sort, restating tf_grouping_g.cu:83-123) and the first k columns.  Returns (val, idx)."""
    x1, x2 = _f(xyz1), _f(xyz2)
    diff = (x1[:, None, :, :] - x2[:, :, None, :]).astype(_F)
    sq = (diff * diff).astype(_F)
    dist = ((sq[..., 0] + sq[..., 1]).astype(_F) + sq[..., 2]).astype(_F)
    outi, out = oracle_selection_sort(k, dist)
    return np.ascontiguousarray(out[:, :, :k]), np.ascontiguousarray(outi[:, :, :k])


# ------------------------------------------------------------------ reference CPU functions
def refcpu_query_ball_point(radius: float, nsample: int, xyz1, xyz2):
    """tf_ops/grouping/test/query_ball_point.cpp:19 (no pts_cnt output). idx pre-zeroed."""
    xyz1, xyz2 = _f(xyz1), _f(xyz2)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    idx = np.zeros((b, m, nsample), _I)
    refcpu()._ZN7ref_qbp20query_ball_point_cpuEiiifiPKfS1_Pi(
        c_int(b), c_int(n), c_int(m), c_float(radius), c_int(nsample), _p(xyz1), _p(xyz2), _p(idx))
    return idx


def refcpu_group_point(points, idx):
    points, idx = _f(points), _i(idx)
    b, n, c = points.shape
    _, m, s = idx.shape
    out = np.empty((b, m, s, c), _F)
    refcpu()._ZN7ref_qbp15group_point_cpuEiiiiiPKfPKiPf(
        c_int(b), c_int(n), c_int(c), c_int(m), c_int(s), _p(points), _p(idx), _p(out))
    return out


def refcpu_group_point_grad(points_shape, idx, grad_out):
    idx, grad_out = _i(idx), _f(grad_out)
    b, n, c = points_shape
    _, m, s = idx.shape
    g = np.zeros((b, n, c), _F)
    refcpu()._ZN7ref_qbp20group_point_grad_cpuEiiiiiPKfPKiPf(
        c_int(b), c_int(n), c_int(c), c_int(m), c_int(s), _p(grad_out), _p(idx), _p(g))
    return g


def refcpu_three_nn(xyz1, xyz2):
    xyz1, xyz2 = _f(xyz1), _f(xyz2)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    dist = np.empty((b, n, 3), _F)
    idx = np.empty((b, n, 3), _I)
    refcpu()._ZN10ref_interp11threenn_cpuEiiiPKfS1_PfPi(
        c_int(b), c_int(n), c_int(m), _p(xyz1), _p(xyz2), _p(dist), _p(idx))
    return dist, idx


def refcpu_three_interpolate(points, idx, weight):
    points, idx, weight = _f(points), _i(idx), _f(weight)
    b, m, c = points.shape
    n = idx.shape[1]
    out = np.empty((b, n, c), _F)
    refcpu()._ZN10ref_interp20threeinterpolate_cpuEiiiiPKfPKiS1_Pf(
        c_int(b), c_int(m), c_int(c), c_int(n), _p(points), _p(idx), _p(weight), _p(out))
    return out


def refcpu_three_interpolate_grad(points_shape, idx, weight, grad_out):
    idx, weight, grad_out = _i(idx), _f(weight), _f(grad_out)
    b, m, c = points_shape
    n = idx.shape[1]
    g = np.zeros((b, m, c), _F)
    refcpu()._ZN10ref_interp25threeinterpolate_grad_cpuEiiiiPKfPKiS1_Pf(
        c_int(b), c_int(n), c_int(c), c_int(m), _p(grad_out), _p(idx), _p(weight), _p(g))
    return g


def refcpu_selection_sort(k: int, dist):
    dist = _f(dist)
    b, m, n = dist.shape
    outi = np.empty((b, m, n), _I)
    out = np.empty((b, m, n), _F)
    refcpu()._ZN9ref_ssort18selection_sort_cpuEiiiiPKfPiPf(
        c_int(b), c_int(n), c_int(m), c_int(k), _p(dist), _p(outi), _p(out))
    return outi, out


# ------------------------------------------------- reference CUDA launchers (torch CUDA tensors)
def _tp(t):
    return c_void_p(t.data_ptr())


def refcuda_fps(npoint: int, xyz):
    """farthestpointsamplingLauncher, tf_sampling_g.cu:203 — needs the 32*n float scratch."""
    import torch
    b, n, _ = xyz.shape
    temp = torch.empty((32, n), dtype=torch.float32, device=xyz.device)
    out = torch.zeros((b, npoint), dtype=torch.int32, device=xyz.device)
    torch.cuda.synchronize()
    refcuda()[0]._Z29farthestpointsamplingLauncheriiiPKfPfPi(
        c_int(b), c_int(n), c_int(npoint), _tp(xyz), _tp(temp), _tp(out))
    torch.cuda.synchronize()
    return out


def refcuda_prob_sample(inp, inpr, return_cumsum: bool = False):
    """probsampleLauncher, tf_sampling_g.cu:198 — needs the b*n float scratch."""
    import torch
    b, n = inp.shape
    m = inpr.shape[1]
    temp = torch.empty((b, n), dtype=torch.float32, device=inp.device)
    out = torch.zeros((b, m), dtype=torch.int32, device=inp.device)
    torch.cuda.synchronize()
    refcuda()[0]._Z18probsampleLauncheriiiPKfS0_PfPi(c_int(b), c_int(n), c_int(m), _tp(inp), _tp(inpr), _tp(temp), _tp(out))
    torch.cuda.synchronize()
    return (out, temp) if return_cumsum else out


def refcuda_gather_point(inp, idx):
    import torch
    b, n, _ = inp.shape
    m = idx.shape[1]
    out = torch.empty((b, m, 3), dtype=torch.float32, device=inp.device)
    torch.cuda.synchronize()
    refcuda()[0]._Z19gatherpointLauncheriiiPKfPKiPf(c_int(b), c_int(n), c_int(m), _tp(inp), _tp(idx), _tp(out))
    torch.cuda.synchronize()
    return out


def refcuda_gather_point_grad(inp_shape, idx, out_g):
    import torch
    b, n, _ = inp_shape
    m = idx.shape[1]
    g = torch.zeros((b, n, 3), dtype=torch.float32, device=idx.device)
    torch.cuda.synchronize()
    refcuda()[0]._Z23scatteraddpointLauncheriiiPKfPKiPf(c_int(b), c_int(n), c_int(m), _tp(out_g), _tp(idx), _tp(g))
    torch.cuda.synchronize()
    return g


def refcuda_query_ball_point(radius: float, nsample: int, xyz1, xyz2):
    """queryBallPointLauncher, tf_grouping_g.cu:125. idx is pre-zeroed (the reference leaves rows
    without a hit uninitialised)."""
    import torch
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    idx = torch.zeros((b, m, nsample), dtype=torch.int32, device=xyz1.device)
    cnt = torch.zeros((b, m), dtype=torch.int32, device=xyz1.device)
    torch.cuda.synchronize()
    refcuda()[1]._Z22queryBallPointLauncheriiifiPKfS0_PiS1_(
        c_int(b), c_int(n), c_int(m), c_float(radius), c_int(nsample), _tp(xyz1), _tp(xyz2), _tp(idx), _tp(cnt))
    torch.cuda.synchronize()
    return idx, cnt


def refcuda_group_point(points, idx):
    import torch
    b, n, c = points.shape
    _, m, s = idx.shape
    out = torch.empty((b, m, s, c), dtype=torch.float32, device=points.device)
    torch.cuda.synchronize()
    refcuda()[1]._Z18groupPointLauncheriiiiiPKfPKiPf(
        c_int(b), c_int(n), c_int(c), c_int(m), c_int(s), _tp(points), _tp(idx), _tp(out))
    torch.cuda.synchronize()
    return out


def refcuda_group_point_grad(points_shape, idx, grad_out):
    import torch
    b, n, c = points_shape
    _, m, s = idx.shape
    g = torch.zeros((b, n, c), dtype=torch.float32, device=idx.device)
    torch.cuda.synchronize()
    refcuda()[1]._Z22groupPointGradLauncheriiiiiPKfPKiPf(
        c_int(b), c_int(n), c_int(c), c_int(m), c_int(s), _tp(grad_out), _tp(idx), _tp(g))
    torch.cuda.synchronize()
    return g


def refcuda_selection_sort(k: int, dist):
    import torch
    b, m, n = dist.shape
    outi = torch.empty((b, m, n), dtype=torch.int32, device=dist.device)
    out = torch.empty((b, m, n), dtype=torch.float32, device=dist.device)
    torch.cuda.synchronize()
    refcuda()[1]._Z21selectionSortLauncheriiiiPKfPiPf(
        c_int(b), c_int(n), c_int(m), c_int(k), _tp(dist), _tp(outi), _tp(out))
    torch.cuda.synchronize()
    return outi, out
