"""Parity at BASELINE.json's own sizes against the reference's own code (VERDICT r1, items 1):
the outputs of the reference CUDA kernels rebuilt for sm_100a and of the reference CPU functions on
these tests' inputs (tests/golden/ref_cuda_cases.npz, a seeded sample of rows per case).  Every index
tensor bit-exact; three_interpolate bit-exact (contract 1e-5)."""
import numpy as np
import pytest
import torch

from conftest import assert_golden_rows, load_golden
from oracle import oracle as O
from pointnet2_b200 import _lib, workloads as W
from pointnet2_b200.tf_grouping import knn_point, query_ball_point
from pointnet2_b200.tf_interpolate import three_interpolate, three_nn, three_nn_interpolate
from pointnet2_b200.tf_sampling import farthest_point_sample, farthest_point_sample_and_gather, gather_point

pytestmark = pytest.mark.gpu


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ---- cfg5: ball query at N = 65536 and 262144, M = N/4, S = 32, r = 0.1 (tf_grouping_g.cu:3-36) ------------
@pytest.mark.parametrize("b,n", [(2, 65536), (1, 262144)])
def test_cfg5_ball_query_matches_reference_kernel(dev, b, n):
    m = n // 4
    x = T(W.cloud_uniform(b, n, 100 + int(np.log2(n))), dev)
    _, nx = farthest_point_sample_and_gather(m, x)
    idx, cnt = query_ball_point(0.1, 32, x, nx)
    g = load_golden("ref_cuda_cases")
    assert_golden_rows(cnt, g, f"cfg5_bq/{b}_{n}", "cnt")
    assert_golden_rows(idx, g, f"cfg5_bq/{b}_{n}", "idx")


def test_cfg5_ball_query_sparse_radius_matches_reference_kernel(dev):
    """Same size with balls that do NOT fill up (r = 0.01: ~1 neighbour), so every query scans its
    whole neighbourhood and the padding path runs on every row."""
    b, n = 1, 65536
    x = T(W.cloud_uniform(b, n, 116), dev)
    nx = x[:, ::4].contiguous()
    idx, cnt = query_ball_point(0.01, 32, x, nx)
    g = load_golden("ref_cuda_cases")
    assert_golden_rows(cnt, g, "cfg5_bq_sparse", "cnt")
    assert_golden_rows(idx, g, "cfg5_bq_sparse", "idx")


# ---- cfg5: FPS at the largest sizes (tf_sampling_g.cu:105-170) ---------------------------------------------
@pytest.mark.parametrize("gen,b,n,m", [("U", 1, 262144, 640), ("D", 2, 262144, 512), ("U", 2, 131073, 512), ("U", 8, 65536, 1024),
                                       ("D", 8, 16384, 2048)])
def test_large_fps_matches_reference_kernel(dev, gen, b, n, m):
    x = T(W.DISTRIBUTIONS[gen](b, n, 118), dev)
    g, case = load_golden("ref_cuda_cases"), f"fps_large/{gen}_{b}_{n}_{m}"
    idx = farthest_point_sample(m, x)
    assert_golden_rows(idx, g, case, "idx")
    fi, fx = farthest_point_sample_and_gather(m, x)
    assert torch.equal(fi, idx)
    assert_golden_rows(fx, g, case, "new_xyz")


def test_eight_clouds_of_262144_points_run_as_co_resident_clusters(dev):
    """8 x 262 144 points: no power-of-two cluster size keeps eight clusters resident on B200 (seven 16-CTA clusters
    fit), so the planner must pick the register + shared-memory kernel with a smaller cluster — and the picks must
    be the ones the one-cloud-at-a-time plan (16-CTA clusters, validated against the reference kernel above) makes."""
    import ctypes
    lib = _lib.load()
    b, n, m = 8, 262144, 48
    t, pp, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    assert lib.pn2_fps_plan(b, n, ctypes.byref(t), ctypes.byref(pp), ctypes.byref(c)) == 0
    assert c.value >= 2 and t.value * pp.value * c.value >= n
    assert lib.pn2_fps_cluster_capacity(t.value, pp.value, c.value) >= b, "planned clusters are not co-resident"
    x = T(np.concatenate([W.cloud_duplicates(4, n, 131), W.cloud_uniform(4, n, 132)]), dev)
    idx, new_xyz = farthest_point_sample_and_gather(m, x)
    for i in range(b):
        one_idx, one_xyz = farthest_point_sample_and_gather(m, x[i:i + 1].contiguous())
        assert torch.equal(idx[i:i + 1], one_idx) and torch.equal(new_xyz[i:i + 1], one_xyz)


# ---- cfg4: the whole FP stack at B = 16 (tf_interpolate.cpp:60-127) ------------------------------------------
def test_cfg4_fp_stack_matches_reference_cpu_functions(dev):
    c4 = W.CFG4_SEMSEG
    b = c4["b"]
    g = load_golden("ref_cuda_cases")
    xyz = W.cloud_duplicates(b, c4["n"], 100)
    x = T(xyz, dev)
    levels = {c4["n"]: x}
    cur = x
    for L in c4["sa"]:  # the real centroid hierarchy 8192 -> 1024 -> 256 -> 64 -> 16
        cur = gather_point(cur, farthest_point_sample(L["npoint"], cur))
        levels[L["npoint"]] = cur
    for F in c4["fp"]:
        n, m, c = F["n"], F["m"], F["c"]
        x1, x2 = levels[n], levels[m]
        p2 = W.features(b, m, c, 105)
        dist, idx = three_nn(x1, x2)
        assert_golden_rows(idx, g, f"cfg4_fp/{n}_{m}", "idx")
        assert_golden_rows(dist, g, f"cfg4_fp/{n}_{m}", "dist")
        d = torch.clamp(dist, min=1e-10)
        w = (1.0 / d) / (1.0 / d).sum(dim=2, keepdim=True)
        out = three_interpolate(T(p2, dev), idx, w)
        assert_golden_rows(out, g, f"cfg4_fp/{n}_{m}", "out")  # bit-exact (contract 1e-5)
        fused = three_nn_interpolate(x1, x2, T(p2, dev))
        assert float((fused - out).abs().max()) <= 1e-5


# ---- n3: knn_point against the reference's composite (tf_grouping.py:48-73 + selection_sort_gpu) -------------
# The reference composite: pairwise squared distances as the reference's graph computes them (tile, subtract,
# square, reduce_sum over the 3 coordinates: each product rounded, summed left to right), then the rebuilt
# selection_sort_gpu; its first k columns are knn_point's outputs (oracle/gen_golden.py: knn_ref).
@pytest.mark.parametrize("gen,b,n,m,k", [("U", 4, 4096, 256, 32), ("D", 3, 3000, 200, 32), ("D", 2, 2048, 128, 128), ("S", 2, 1024, 512, 16),
                                         ("U", 2, 40, 10, 40), ("U", 2, 70, 10, 64), ("D", 2, 700, 64, 1), ("U", 1, 8192, 128, 3)])
def test_knn_point_matches_reference_composite(dev, gen, b, n, m, k):
    xyz = W.DISTRIBUTIONS[gen](b, n, 120)
    x1 = T(xyz, dev)
    x2 = gather_point(x1, farthest_point_sample(m, x1)) if gen != "U" else T(W.cloud_uniform(b, m, 121), dev)
    val, idx = knn_point(k, x1, x2)
    g, case = load_golden("ref_cuda_cases"), f"knn/{gen}_{b}_{n}_{m}_{k}"
    assert_golden_rows(idx, g, case, "idx")
    assert_golden_rows(val, g, case, "val")
    with pytest.raises(ValueError):
        knn_point(n + 1, x1, x2)


@pytest.mark.parametrize("k", [4, 32, 48])
def test_knn_point_with_nan_and_inf_points_matches_the_selection_sort(dev, k):
    """Non-finite distances: the selection sort starts every round from min = v[s] and replaces it by strict '<'
    (tf_grouping_g.cu:98-108), so a NaN at a position < k is output in its own round and a NaN anywhere else is
    never taken; inf is an ordinary (largest) value.  Checked against the CPU restatement of the composite."""
    b, n, m = 3, 300, 40
    xyz = W.cloud_uniform(b, n, 123)
    xyz[0, 2, 1] = np.nan      # inside the first k positions
    xyz[0, 150, 0] = np.nan    # beyond them
    xyz[1, 1, 2] = np.inf
    xyz[1, 200, 0] = -np.inf
    xyz[2, k + 1, 0] = np.nan  # among the first candidates of the top-k list
    q = W.cloud_uniform(b, m, 124)
    val, idx = knn_point(k, T(xyz, dev), T(q, dev))
    wv, wi = O.oracle_knn_point(k, xyz, q)
    np.testing.assert_array_equal(idx.cpu().numpy(), wi)
    np.testing.assert_array_equal(val.cpu().numpy(), wv)


def test_knn_point_full_size_matches_reference_composite(dev):
    """(32, 1024, 4096, k = 32) — cfg2's shape (the reference composite ran in 4 slices of 8 clouds so
    that its (b,m,n) matrices stay below 1 GB)."""
    xyz = W.cloud_duplicates(32, 4096, 122)  # ties everywhere
    x1 = T(xyz, dev)
    x2 = gather_point(x1, farthest_point_sample(1024, x1))
    val, idx = knn_point(32, x1, x2)
    g = load_golden("ref_cuda_cases")
    assert_golden_rows(idx, g, "knn_full", "idx")
    assert_golden_rows(val, g, "knn_full", "val")
