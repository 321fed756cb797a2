"""GPU tests of the round-2 feature-propagation / grouping-tail kernels:
  * pn2_fp_interpolate_concat (multi-lane 3-NN + weights + interpolation + concat with points1) against
    the unfused op sequence and the reference's CPU functions;
  * pn2_three_interpolate_grad_det (inverse index, ordered sums) bit-exact against threeinterpolate_grad_cpu;
  * the flat 32-row group_concat kernel at the reference networks' odd row widths (67, 131, 259, 323)."""
import numpy as np
import pytest
import torch

from conftest import assert_golden_rows, load_golden
from oracle import oracle as O
from pointnet2_b200 import _lib, tf_interpolate as TI, workloads as W
from pointnet2_b200.pointnet_util import group_and_concat, pointnet_fp_module
from pointnet2_b200.tf_grouping import group_point, query_ball_point
from pointnet2_b200.tf_interpolate import fp_interpolate_concat, three_interpolate, three_nn, three_nn_interpolate

pytestmark = pytest.mark.gpu


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def unfused_fp(x1, x2, p1, p2):
    dist, idx = three_nn(x1, x2)
    d = torch.clamp(dist, min=1e-10)
    w = (1.0 / d) / (1.0 / d).sum(dim=2, keepdim=True)
    out = three_interpolate(p2, idx, w)
    return out if p1 is None else torch.cat([out, p1], dim=2)


# (b, n, m, c2, c1): every lanes-per-point regime (G = 1 .. 32), vector and scalar widths, m < 3
FP_CASES = [(16, 64, 16, 512, 256), (16, 256, 64, 256, 128), (16, 1024, 256, 256, 64), (4, 8192, 1024, 128, 0), (2, 8192, 1024, 128, 32),
            (2, 77, 9, 5, 3), (3, 300, 2, 8, 0), (2, 50, 1, 4, 4), (1, 5, 700, 64, 64), (2, 4000, 3000, 12, 0), (1, 33, 130, 7, 0)]


@pytest.mark.parametrize("b,n,m,c2,c1", FP_CASES)
def test_fp_interpolate_concat_matches_unfused(dev, b, n, m, c2, c1):
    x1, x2 = T(W.cloud_uniform(b, n, 201), dev), T(W.cloud_uniform(b, m, 202), dev)
    p2 = T(W.features(b, m, c2, 203), dev)
    p1 = T(W.features(b, n, c1, 204), dev) if c1 else None
    got = fp_interpolate_concat(x1, x2, p1, p2)
    want = unfused_fp(x1, x2, p1, p2)
    # neighbours and distances are bit-exact; the weights' 3-term sum is (r1+r2)+r3 here and whatever order torch's
    # reduction uses in the unfused path, so the interpolated half is compared at the contract's 1e-5 ...
    assert float((got[..., :c2] - want[..., :c2]).abs().max()) <= 1e-5 * max(1.0, float(want[..., :c2].abs().max()))
    if c1:
        assert torch.equal(got[..., c2:], p1)  # ... and the concatenated half is a copy
    assert torch.equal(pointnet_fp_module(x1, x2, p1, p2), got)
    out, d, i, w = three_nn_interpolate(x1, x2, p2, return_aux=True)
    wd, wi = three_nn(x1, x2)
    assert torch.equal(d, wd) and torch.equal(i, wi)
    # with the kernel's own weights the interpolation is bit-exact against the stand-alone op (and the oracle)
    assert torch.equal(out, three_interpolate(p2, i, w)) and torch.equal(out, got[..., :c2])


def test_fp_interpolate_concat_with_duplicate_known_points(dev):
    """Ties between known points at equal distance: the multi-lane merge must keep the lower index
    (tf_interpolate.cpp:74-89 strict '<' over ascending k)."""
    b, n, m = 2, 200, 96
    x2 = W.cloud_duplicates(b, m, 205)
    x1 = np.concatenate([x2[:, ::2], W.cloud_uniform(b, n - m // 2, 206)], axis=1).astype(np.float32)
    p2 = W.features(b, m, 16, 207)
    rd, ri = O.oracle_three_nn(x1, x2)
    out, d, i, w = three_nn_interpolate(T(x1, dev), T(x2, dev), T(p2, dev), return_aux=True)
    np.testing.assert_array_equal(i.cpu().numpy(), ri)
    np.testing.assert_array_equal(d.cpu().numpy(), rd)


# ------------------------------------------------------------------------------------------- deterministic gradient
GRAD_CASES = [(16, 8192, 1024, 128), (4, 1024, 256, 256), (2, 300, 40, 7), (2, 64, 16, 512), (3, 500, 1, 8), (2, 500, 2, 33), (1, 20000, 5, 16),
              (2, 10, 300, 4), (2, 3000, 60, 132)]


@pytest.mark.parametrize("b,n,m,c", GRAD_CASES)
def test_three_interpolate_grad_deterministic_matches_reference_order(dev, b, n, m, c):
    lib = _lib.load()
    x1, x2 = W.cloud_uniform(b, n, 211), W.cloud_uniform(b, m, 212)
    _, idx = O.oracle_three_nn(x1, x2)
    w = np.random.RandomState(213).random_sample((b, n, 3)).astype(np.float32)
    go = W.features(b, n, c, 214)
    want = O.oracle_three_interpolate_grad((b, m, c), idx, w, go)  # the C restatement adds in the reference's (j, t) order
    assert_golden_rows(want, load_golden("ref_cpu_cases"), f"three_interp_grad_det/{b}_{n}_{m}_{c}", "out")
    gp = torch.full((b, m, c), 7.0, dtype=torch.float32, device=dev)  # no zero-fill needed: overwritten
    wsb = int(lib.pn2_three_interpolate_grad_det_workspace_bytes(b, n, m))
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    tg, ti, tw = T(go, dev), T(idx, dev), T(w, dev)
    # lists of up to 256 (j, t) entries are summed in the reference's order: bit-exact.  Longer ones (degenerate layers:
    # m < 3, ...) are summed in 8 ordered pieces: deterministic, equal up to rounding.
    longest = max(int(np.bincount(idx[i].ravel(), minlength=m).max()) for i in range(b))
    runs = []
    for _ in range(2):
        rc = lib.pn2_three_interpolate_grad_det(b, n, c, m, tg.data_ptr(), ti.data_ptr(), tw.data_ptr(), gp.data_ptr(), ws.data_ptr(), wsb, None)
        assert rc == 0
        torch.cuda.synchronize()
        runs.append(gp.cpu().numpy().copy())
        gp.fill_(7.0)
    np.testing.assert_array_equal(runs[0], runs[1])  # run-to-run deterministic, always
    if longest <= 256:
        np.testing.assert_array_equal(runs[0], want)
    else:
        np.testing.assert_allclose(runs[0], want, rtol=2e-5, atol=2e-5 * float(np.abs(want).max()))
    # and through autograd (the default backward)
    p = T(W.features(b, m, c, 215), dev).requires_grad_(True)
    (three_interpolate(p, ti, tw) * tg).sum().backward()
    np.testing.assert_array_equal(p.grad.cpu().numpy(), runs[0])
    TI.DETERMINISTIC_GRAD = False
    try:
        p2 = p.detach().clone().requires_grad_(True)
        (three_interpolate(p2, ti, tw) * tg).sum().backward()
    finally:
        TI.DETERMINISTIC_GRAD = True
    scale = max(1.0, float(np.abs(want).max()))
    assert float((p2.grad - p.grad).abs().max()) <= 1e-4 * scale  # the atomic path: the reference's own bar


# ------------------------------------------------------------------------------------------- group_concat at odd widths
@pytest.mark.parametrize("xyz_first", [True, False])
@pytest.mark.parametrize("b,n,m,s,c", [(16, 1024, 256, 32, 64), (16, 256, 64, 32, 128), (4, 64, 16, 32, 256), (8, 512, 128, 64, 320),
                                       (2, 700, 33, 7, 5), (1, 100, 3, 2, 1), (2, 300, 50, 33, 13)])
def test_group_concat_flat_kernel_matches_separate_ops(dev, b, n, m, s, c, xyz_first):
    xyz = T(W.cloud_uniform(b, n, 221), dev)
    feats = T(W.features(b, n, c, 222), dev)
    nx = xyz[:, :m].contiguous()
    idx, _ = query_ball_point(0.3, s, xyz, nx)
    got, gx = group_and_concat(xyz, nx, feats, idx, xyz_first=xyz_first)
    wx = group_point(xyz, idx) - nx.unsqueeze(2)
    wf = group_point(feats, idx)
    want = torch.cat([wx, wf] if xyz_first else [wf, wx], dim=-1)
    assert torch.equal(gx, wx)
    assert torch.equal(got, want)
