"""GPU tests of 16-bit features (bfloat16 / float16) through the grouping and interpolation ops: gathers and concats
copy bits, interpolation equals the float32 op on the widened features rounded once, gradients accumulate in float32
and come back in the feature dtype, and the networks train under torch.autocast."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from pointnet2_b200 import _lib, nets, tf_interpolate, workloads as W
from pointnet2_b200.pointnet_util import (group_and_concat, pointnet_fp_module, pointnet_sa_module,
                                          pointnet_sa_module_msg)
from pointnet2_b200.tf_grouping import group_point, query_ball_point
from pointnet2_b200.tf_interpolate import fp_interpolate_concat, three_interpolate, three_nn, three_nn_interpolate

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HALF = [torch.bfloat16, torch.float16]


def bits_equal(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    if a.dtype in HALF:
        return torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16))
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def _weights(xyz1, xyz2):
    dist, idx = three_nn(xyz1, xyz2)
    dist = torch.clamp(dist, min=1e-10)
    norm = (1.0 / dist).sum(dim=2, keepdim=True)
    return idx, (1.0 / dist) / norm


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [1, 2, 3, 7, 8, 64, 67, 128, 131, 259, 320, 323])
def test_group_point_copies_bits(dev, dt, c):
    g = _gen(dev, c)
    b, n, m, s = 3, 257, 40, 16
    points = (torch.randn((b, n, c), device=dev, generator=g) * 3).to(dt)
    idx = torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)
    out = group_point(points, idx)
    want = points[torch.arange(b, device=dev).view(b, 1, 1), idx.long()]
    assert bits_equal(out, want)


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [8, 64, 67, 320])
def test_group_point_at_a_2_byte_offset(dev, dt, c):
    g = _gen(dev, 100 + c)
    b, n, m, s = 2, 129, 33, 8
    store = (torch.randn(b * n * c + 1, device=dev, generator=g)).to(dt)
    points = store[1:].view(b, n, c)  # contiguous view, 2 bytes past a 16-byte boundary
    assert points.is_contiguous() and points.data_ptr() % 16 == 2
    idx = torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)
    assert bits_equal(group_point(points, idx), points[torch.arange(b, device=dev).view(b, 1, 1), idx.long()])
    xyz = torch.rand((b, n, 3), device=dev, generator=g)
    new_xyz = torch.rand((b, m, 3), device=dev, generator=g)
    out, _ = group_and_concat(xyz, new_xyz, points, idx, xyz_first=True)
    bi = torch.arange(b, device=dev).view(b, 1, 1)
    want = torch.cat([(xyz[bi, idx.long()] - new_xyz.unsqueeze(2)).to(dt), points[bi, idx.long()]], -1)
    assert bits_equal(out, want)


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [3, 8, 131])
def test_gathers_keep_nan_inf_and_negative_zero(dev, dt, c):
    b, n, m, s = 2, 64, 16, 8
    g = _gen(dev, 7)
    raw = torch.randint(-32768, 32767, (b, n, c), device=dev, generator=g, dtype=torch.int16)
    raw[:, :8] = torch.tensor([0x7FC1, 0xFFC3, 0x7F81, 0x7C01, 0x7F80, 0xFF80, -32768, 0x7E12],
                              dtype=torch.int32, device=dev).to(torch.int16).view(1, 8, 1)
    points = raw.view(dt)
    idx = torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)
    idx[:, :, :4] = torch.arange(4, device=dev, dtype=torch.int32)
    bi = torch.arange(b, device=dev).view(b, 1, 1)
    assert bits_equal(group_point(points, idx), points[bi, idx.long()])
    xyz = torch.rand((b, n, 3), device=dev, generator=g)
    new_xyz = torch.rand((b, m, 3), device=dev, generator=g)
    out, _ = group_and_concat(xyz, new_xyz, points, idx, xyz_first=False)
    assert bits_equal(out[..., :c], points[bi, idx.long()])


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [0, 3, 8, 64, 67, 128, 320])
@pytest.mark.parametrize("xyz_first", [True, False])
def test_group_and_concat(dev, dt, c, xyz_first):
    g = _gen(dev, 3 * c + xyz_first)
    b, n, m, s = 3, 300, 50, 16
    xyz = torch.rand((b, n, 3), device=dev, generator=g)
    new_xyz = torch.rand((b, m, 3), device=dev, generator=g)
    points = torch.randn((b, n, c), device=dev, generator=g).to(dt) if c else None
    idx = torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)
    out, gxyz = group_and_concat(xyz, new_xyz, points, idx, xyz_first=xyz_first)
    bi = torch.arange(b, device=dev).view(b, 1, 1)
    centred = xyz[bi, idx.long()] - new_xyz.unsqueeze(2)
    if points is None:
        assert out.dtype == torch.float32 and bits_equal(out, centred)
        return
    feats = points[bi, idx.long()]
    parts = [centred.to(dt), feats] if xyz_first else [feats, centred.to(dt)]
    assert bits_equal(out, torch.cat(parts, -1))
    assert gxyz.dtype == torch.float32
    _, gxyz32 = group_and_concat(xyz, new_xyz, points.float(), idx, xyz_first=xyz_first)
    assert bits_equal(gxyz, gxyz32)


@pytest.mark.parametrize("dt", HALF)
def test_half_coordinates_and_weights_are_refused(dev, dt):
    x = torch.rand((1, 16, 3), device=dev)
    f = torch.randn((1, 16, 8), device=dev).to(dt)
    idx = torch.zeros((1, 4, 2), dtype=torch.int32, device=dev)
    with pytest.raises(TypeError):
        group_and_concat(x, x.to(dt), f, idx)
    with pytest.raises(TypeError):
        fp_interpolate_concat(x, x.to(dt), None, f)
    with pytest.raises(TypeError):
        three_nn_interpolate(x, x.to(dt), f)
    i3, w = _weights(x, x)
    with pytest.raises(TypeError):
        three_interpolate(f, i3, w.to(dt))
    with pytest.raises(TypeError):
        fp_interpolate_concat(x, x, f.float(), f)


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [1, 5, 8, 64, 67, 128])
def test_three_interpolate_is_the_float32_op_rounded_once(dev, dt, c):
    g = _gen(dev, 40 + c)
    b, n, m = 2, 1000, 130
    xyz1 = torch.rand((b, n, 3), device=dev, generator=g)
    xyz2 = torch.rand((b, m, 3), device=dev, generator=g)
    points = torch.randn((b, m, c), device=dev, generator=g).to(dt)
    idx, w = _weights(xyz1, xyz2)
    out = three_interpolate(points, idx, w)
    assert bits_equal(out, three_interpolate(points.float(), idx, w).to(dt))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c2,c1", [(8, 0), (64, 0), (67, 0), (128, 64), (128, 3), (5, 8), (256, 128)])
@pytest.mark.parametrize("n,m", [(64, 16), (2048, 512)])
def test_fused_fp_front_end(dev, dt, c2, c1, n, m):
    g = _gen(dev, c2 * 7 + c1 + n)
    b = 2
    xyz1 = torch.rand((b, n, 3), device=dev, generator=g)
    xyz2 = torch.rand((b, m, 3), device=dev, generator=g)
    p2 = torch.randn((b, m, c2), device=dev, generator=g).to(dt)
    p1 = torch.randn((b, n, c1), device=dev, generator=g).to(dt) if c1 else None
    out = fp_interpolate_concat(xyz1, xyz2, p1, p2)
    want = fp_interpolate_concat(xyz1, xyz2, None if p1 is None else p1.float(), p2.float()).to(dt)
    assert bits_equal(out, want)
    if c1 == 0:
        o, d, i, w = three_nn_interpolate(xyz1, xyz2, p2, return_aux=True)
        o32, d32, i32, w32 = three_nn_interpolate(xyz1, xyz2, p2.float(), return_aux=True)
        assert bits_equal(o, o32.to(dt)) and bits_equal(d, d32) and torch.equal(i, i32) and bits_equal(w, w32)
        assert bits_equal(three_nn_interpolate(xyz1, xyz2, p2), o)


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [5, 64, 128])
def test_three_interpolate_gradients(dev, dt, c):
    g = _gen(dev, 70 + c)
    b, n, m = 2, 2048, 256
    xyz1 = torch.rand((b, n, 3), device=dev, generator=g)
    xyz2 = torch.rand((b, m, 3), device=dev, generator=g)
    idx, w = _weights(xyz1, xyz2)
    grad_out = torch.randn((b, n, c), device=dev, generator=g).to(dt)
    saved = tf_interpolate.DETERMINISTIC_GRAD
    try:
        tf_interpolate.DETERMINISTIC_GRAD = True
        p = torch.zeros((b, m, c), device=dev, dtype=dt, requires_grad=True)
        three_interpolate(p, idx, w).backward(grad_out)
        p32 = torch.zeros((b, m, c), device=dev, requires_grad=True)
        three_interpolate(p32, idx, w).backward(grad_out.float())
        assert p.grad.dtype == dt and bits_equal(p.grad, p32.grad.to(dt))
        tf_interpolate.DETERMINISTIC_GRAD = False
        q = torch.zeros((b, m, c), device=dev, dtype=dt, requires_grad=True)
        three_interpolate(q, idx, w).backward(grad_out)
    finally:
        tf_interpolate.DETERMINISTIC_GRAD = saved
    flat = (torch.arange(b, device=dev).view(b, 1, 1) * m + idx.long()).view(-1)
    contrib = (grad_out.double().unsqueeze(2) * w.double().unsqueeze(3)).view(-1, c)
    want = torch.zeros((b * m, c), device=dev, dtype=torch.float64).index_add_(0, flat, contrib)
    assert q.grad.dtype == dt
    # float32 accumulation of <= a few dozen terms, then one rounding to dt
    tol = torch.finfo(dt).eps * want.abs() + 1e-4 * (1 + want.abs())
    assert bool(((q.grad.double().view(-1, c) - want).abs() <= tol).all())


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("c", [3, 8, 67, 128])
def test_group_gradients(dev, dt, c):
    g = _gen(dev, 90 + c)
    b, n, m, s = 2, 200, 64, 16
    idx = torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)
    grad_out = torch.randn((b, m, s, c), device=dev, generator=g).to(dt)
    p = torch.zeros((b, n, c), device=dev, dtype=dt, requires_grad=True)
    group_point(p, idx).backward(grad_out)
    flat = (torch.arange(b, device=dev).view(b, 1, 1) * n + idx.long()).view(-1)
    want = torch.zeros((b * n, c), device=dev, dtype=torch.float64).index_add_(0, flat, grad_out.double().view(-1, c))
    tol = torch.finfo(dt).eps * want.abs() + 1e-4 * (1 + want.abs())
    assert p.grad.dtype == dt and bool(((p.grad.double().view(-1, c) - want).abs() <= tol).all())
    # the concat's feature part and its float32 coordinate part
    xyz = torch.rand((b, n, 3), device=dev, generator=g, requires_grad=True)
    new_xyz = torch.rand((b, m, 3), device=dev, generator=g)
    q = torch.zeros((b, n, c), device=dev, dtype=dt, requires_grad=True)
    for xyz_first in (True, False):
        q.grad, xyz.grad = None, None
        out, _ = group_and_concat(xyz, new_xyz, q, idx, xyz_first=xyz_first)
        go = torch.randn(out.shape, device=dev, generator=g).to(dt)
        out.backward(go)
        feat = go[..., 3:] if xyz_first else go[..., :c]
        gx = (go[..., :3] if xyz_first else go[..., c:]).float()
        want = torch.zeros((b * n, c), device=dev, dtype=torch.float64).index_add_(0, flat, feat.double().reshape(-1, c))
        tol = torch.finfo(dt).eps * want.abs() + 1e-4 * (1 + want.abs())
        assert q.grad.dtype == dt and bool(((q.grad.double().view(-1, c) - want).abs() <= tol).all())
        want_x = torch.zeros((b * n, 3), device=dev, dtype=torch.float64).index_add_(0, flat, gx.double().reshape(-1, 3))
        assert xyz.grad.dtype == torch.float32
        assert torch.allclose(xyz.grad.double().view(-1, 3), want_x, rtol=1e-5, atol=1e-4)


def _cloud(dev, b, n, c, dt, seed):
    xyz = torch.from_numpy(W.cloud_uniform(b, n, seed)).to(dev)
    feats = torch.randn((b, n, c), device=dev, generator=_gen(dev, seed)).to(dt)
    return xyz, feats


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("knn,use_xyz", [(False, True), (False, False), (True, True), (True, False)])
def test_sa_module_without_mlp(dev, dt, knn, use_xyz):
    xyz, f = _cloud(dev, 2, 1024, 64, dt, 11)
    nx, np_, idx = pointnet_sa_module(xyz, f, 128, 0.2, 32, knn=knn, use_xyz=use_xyz)
    nx32, np32, idx32 = pointnet_sa_module(xyz, f.float(), 128, 0.2, 32, knn=knn, use_xyz=use_xyz)
    assert torch.equal(idx, idx32) and bits_equal(nx, nx32)
    assert bits_equal(np_, np32.to(dt))


@pytest.mark.parametrize("dt", HALF)
def test_sa_module_msg_without_mlp(dev, dt):
    xyz, f = _cloud(dev, 2, 1024, 32, dt, 12)
    nx, np_ = pointnet_sa_module_msg(xyz, f, 128, [0.1, 0.2, 0.4], [16, 32, 64])
    nx32, np32 = pointnet_sa_module_msg(xyz, f.float(), 128, [0.1, 0.2, 0.4], [16, 32, 64])
    assert bits_equal(nx, nx32) and bits_equal(np_, np32.to(dt))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("with_points1", [True, False])
def test_fp_module_without_mlp(dev, dt, fused, with_points1):
    xyz1, p1 = _cloud(dev, 2, 1024, 32, dt, 13)
    xyz2, p2 = _cloud(dev, 2, 256, 64, dt, 14)
    p1 = p1 if with_points1 else None
    out = pointnet_fp_module(xyz1, xyz2, p1, p2, fused=fused)
    want = pointnet_fp_module(xyz1, xyz2, None if p1 is None else p1.float(), p2.float(), fused=fused).to(dt)
    assert bits_equal(out, want)
    if p1 is not None:  # mixed feature dtypes take the unfused branch, where torch.cat promotes
        mixed = pointnet_fp_module(xyz1, xyz2, p1.float(), p2, fused=fused)
        assert mixed.dtype == torch.float32 and bits_equal(mixed, torch.cat([want[..., :64].float(), p1.float()], -1))


@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("name,b,n,out", [("cls_ssg", 4, 1024, (4, 40)), ("cls_msg", 3, 1024, (3, 40)),
                                          ("sem_seg", 2, 2048, (2, 2048, 21))])
def test_networks_train_under_autocast(dev, dt, name, b, n, out):
    torch.manual_seed(0)
    net = {"cls_ssg": nets.PointNet2ClsSSG, "cls_msg": nets.PointNet2ClsMSG, "sem_seg": nets.PointNet2SemSeg}[name]().to(dev)
    xyz = torch.from_numpy(W.cloud_surface(b, n, 400)).to(dev)
    with torch.autocast("cuda", dtype=dt):
        pred, _ = net(xyz)
        loss = pred.float().square().mean()
    assert tuple(pred.shape) == out and bool(torch.isfinite(pred).all())
    loss.backward()
    bad = [k for k, p in net.named_parameters() if p.grad is None or not bool(torch.isfinite(p.grad).all())]
    assert not bad, bad
    first = next(net.parameters())
    assert float(first.grad.abs().sum()) > 0


def test_bf16_autocast_training_reduces_the_loss_on_synthetic_shapes(dev):
    spec = importlib.util.spec_from_file_location("train_ddp_demo", os.path.join(ROOT, "tools", "train_ddp_demo.py"))
    demo = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(demo)
    torch.manual_seed(0)
    net = nets.PointNet2ClsSSG(3).to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    rs = np.random.RandomState(7)
    losses = []
    for _ in range(24):
        xyz, lab = demo.synthetic_shapes(16, 512, 3, rs)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            pred, _ = net(torch.from_numpy(xyz).to(dev))
            loss = nets.cls_loss(pred.float(), torch.from_numpy(lab).to(dev))
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    assert np.mean(losses[-6:]) < 0.7 * np.mean(losses[:6]), losses


@pytest.mark.parametrize("dt", HALF)
def test_float32_calls_keep_their_launch_counts(dev, dt):
    """A float32 call issues the launches it always did; the 16-bit call of the same op the same number."""
    xyz, f = _cloud(dev, 2, 512, 64, dt, 15)
    idx, _ = query_ball_point(0.2, 16, xyz, xyz[:, :64].contiguous())
    for fn in (lambda p: group_point(p, idx), lambda p: group_and_concat(xyz, xyz[:, :64].contiguous(), p, idx)):
        torch.cuda.synchronize()
        a = _lib.launch_count(); fn(f.float()); b32 = _lib.launch_count() - a
        a = _lib.launch_count(); fn(f); b16 = _lib.launch_count() - a
        assert b32 == 1 and b16 == 1


def test_group_point_beyond_2_to_31_elements(dev):
    free, _ = torch.cuda.mem_get_info(dev)
    if free < 40 * (1 << 30):
        pytest.skip("needs 40 GiB of free device memory")
    for c, s in ((3, 22000), (8, 8400)):  # the 2-byte row kernel, and the float4 kernel on reinterpreted rows
        b, n, m = 2, 1536, 16384
        g = _gen(dev, c)
        points = torch.randn((b, n, c), device=dev, generator=g).to(torch.bfloat16)
        idx = torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)
        out = group_point(points, idx)
        assert out.numel() > (1 << 31)
        total = b * m * s
        rows = torch.cat([torch.randint(0, total, (200000,), device=dev, generator=g),
                          torch.arange(total - 1000, total, device=dev)])
        want = points[rows // (m * s), idx.view(-1)[rows].long()]
        assert bits_equal(out.view(-1, c)[rows], want)
        del out, idx, points
        torch.cuda.empty_cache()
