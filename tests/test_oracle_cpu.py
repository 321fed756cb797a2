"""CPU tests of the oracle itself (no GPU): the C restatement against the reference's own CPU
functions (their outputs on these very inputs, tests/golden/ref_cpu_cases.npz), the literal FPS
restatement against its closed-form selection order, and the reference's known-answer case."""
import numpy as np
import pytest

from conftest import assert_golden_rows, load_golden
from oracle import oracle as O
from pointnet2_b200 import workloads as W


# ---------------------------------------------------------------- FPS restatement
@pytest.mark.parametrize("gen,b,n,m", [("U", 3, 700, 200), ("D", 2, 1500, 700), ("S", 2, 333, 100), ("U", 2, 40, 64)])
def test_fps_literal_equals_keyorder(gen, b, n, m):
    xyz = W.DISTRIBUTIONS[gen](b, n, 7)
    a = O.oracle_fps(m, xyz)
    k = O.oracle_fps(m, xyz, keyorder=True)
    assert a.dtype == np.int32 and a.shape == (b, m)
    np.testing.assert_array_equal(a, k)
    assert (a[:, 0] == 0).all()


def test_fps_tie_break_prefers_lower_slot_not_lower_index():
    # SURVEY.md Appendix A.1: duplicates at k=2 and k=513 -> the reference returns 513
    # (slot 513 % 512 = 1 beats slot 2).
    n = 600
    xyz = np.zeros((1, n, 3), np.float32)
    xyz[0, :, 0] = np.linspace(0.0, 0.1, n)  # everything close to the origin
    far = np.array([5.0, 5.0, 5.0], np.float32)
    xyz[0, 2] = far
    xyz[0, 513] = far
    idx = O.oracle_fps(2, xyz)
    assert idx[0, 1] == 513
    assert O.oracle_fps(2, xyz, keyorder=True)[0, 1] == 513


def test_fps_cfg1_plumbing():
    c = W.CFG1_FPS_CPU
    xyz = W.cloud_uniform(c["b"], c["n"], c["seed"])
    idx = O.oracle_fps(c["npoint"], xyz)
    assert idx.shape == (8, 512) and idx.dtype == np.int32
    assert (idx[:, 0] == 0).all()
    for r in idx:
        assert len(set(r.tolist())) == 512  # distinct points -> distinct picks
    assert idx.min() >= 0 and idx.max() < 1024


def test_fps_exhausted_points_emit_index_zero():
    xyz = W.cloud_uniform(1, 10, 3)
    idx = O.oracle_fps(16, xyz)
    assert sorted(idx[0, :10].tolist()) == list(range(10))
    assert (idx[0, 10:] == 0).all()


# ---------------------------------------------------------------- vs the reference's CPU code
@pytest.mark.parametrize("r,s", [(0.1, 32), (0.4, 16), (0.05, 8)])
def test_ball_query_nofma_equals_reference_cpu(r, s):
    xyz = W.cloud_uniform(3, 800, 11)
    new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(100, xyz))
    idx, cnt = O.oracle_query_ball_point(r, s, xyz, new_xyz, use_fma=False)
    assert_golden_rows(idx, load_golden("ref_cpu_cases"), f"bq_nofma/{r}_{s}", "idx")
    assert ((cnt >= 1) & (cnt <= s)).all()  # the centroid itself is always inside its ball


def test_group_point_and_grad_equal_reference_cpu():
    g = load_golden("ref_cpu_cases")
    xyz = W.cloud_uniform(2, 500, 12)
    feats = W.features(2, 500, 7, 13)
    new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(64, xyz))
    idx, _ = O.oracle_query_ball_point(0.2, 16, xyz, new_xyz)
    assert_golden_rows(O.oracle_group_point(feats, idx), g, "group", "out")
    go = W.features(2, 64 * 16, 7, 14).reshape(2, 64, 16, 7)
    assert_golden_rows(O.oracle_group_point_grad(feats.shape, idx, go), g, "group_grad", "out")


@pytest.mark.parametrize("n,m,dup", [(600, 150, False), (400, 100, True), (30, 2, False), (10, 1, False)])
def test_three_nn_equals_reference_cpu(n, m, dup):
    g = load_golden("ref_cpu_cases")
    xyz1 = W.cloud_duplicates(2, n, 15, drop=False) if dup else W.cloud_uniform(2, n, 15)
    xyz2 = xyz1[:, :m].copy() if dup else W.cloud_uniform(2, m, 16)
    d, i = O.oracle_three_nn(xyz1, xyz2)
    assert_golden_rows(d, g, f"three_nn/{n}_{m}_{dup}", "dist")
    assert_golden_rows(i, g, f"three_nn/{n}_{m}_{dup}", "idx")
    assert (d[:, :, 0] <= d[:, :, 1]).all() and (d[:, :, 1] <= d[:, :, 2]).all()
    if m < 3:
        assert np.isinf(d[:, :, m:]).all() and (i[:, :, m:] == 0).all()


def test_three_interpolate_and_grad_equal_reference_cpu():
    g = load_golden("ref_cpu_cases")
    xyz1, xyz2 = W.cloud_uniform(2, 300, 17), W.cloud_uniform(2, 60, 18)
    pts = W.features(2, 60, 33, 19)
    d, i = O.oracle_three_nn(xyz1, xyz2)
    dd = np.maximum(d, 1e-10)
    w = ((1.0 / dd) / (1.0 / dd).sum(axis=2, keepdims=True)).astype(np.float32)
    assert_golden_rows(O.oracle_three_interpolate(pts, i, w), g, "three_interp", "out")
    go = W.features(2, 300, 33, 20)
    assert_golden_rows(O.oracle_three_interpolate_grad(pts.shape, i, w, go), g, "three_interp_grad", "out")


def test_selection_sort_known_answer():
    # the reference's only known-answer case, tf_ops/grouping/test/selection_sort.cpp:68-92:
    # dist = 10 - i, b=2, n=4, m=2, k=3 -> idx rows 3 2 1 0
    dist = np.tile(10.0 - np.arange(4, dtype=np.float32), (2, 2, 1))
    outi, out = O.oracle_selection_sort(3, dist)
    assert (outi == np.array([3, 2, 1, 0], np.int32)).all()
    assert (out == np.array([7, 8, 9, 10], np.float32)).all()


def test_selection_sort_topk_is_sorted_prefix():
    dist = np.random.RandomState(21).random_sample((2, 5, 64)).astype(np.float32)
    outi, out = O.oracle_selection_sort(9, dist)
    np.testing.assert_array_equal(out[:, :, :9], np.sort(dist, axis=2)[:, :, :9])
    np.testing.assert_array_equal(np.take_along_axis(dist, outi.astype(np.int64), 2), out)
    assert (np.sort(outi, axis=2) == np.arange(64)).all()  # a permutation


# ---------------------------------------------------------------- threshold trick
@pytest.mark.parametrize("r", [0.1, 0.2, 0.4, 0.8, 1e-3, 3.0, 0.15, 1e-19, 1e30])
def test_ball_threshold_is_exact_boundary(r):
    T = np.float32(O.oracle_ball_threshold(r))
    rf = np.float32(r)
    assert np.sqrt(T, dtype=np.float32) < rf
    nxt = np.nextafter(T, np.float32(np.inf))
    assert not (np.sqrt(nxt, dtype=np.float32) < rf) or nxt == np.float32(np.inf)


def test_ball_threshold_degenerate_radius():
    assert O.oracle_ball_threshold(1e-21) < 0
    assert O.oracle_ball_threshold(1e-20) < 0


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 8, 9, 63, 100, 1000, 8191, 8192, 8193, 20001])
def test_prob_sample_restatement_is_an_inverse_cdf(n):
    """oracle_prob_sample: a monotone float32 cumulative sum close to the float64 one, and the
    lower-bound index of u*total in it (tf_sampling_g.cu:7-104)."""
    rng = np.random.RandomState(n)
    p = rng.random_sample((3, n)).astype(np.float32)
    r = rng.random_sample((3, 40)).astype(np.float32)
    r[:, 0], r[:, 1] = 0.0, 1.0
    c = O.oracle_prob_cumsum(p)
    ref = np.cumsum(p.astype(np.float64), axis=1)
    assert np.abs(c - ref).max() <= 4e-7 * ref.max()
    assert (c[:, 1:] >= c[:, :-1]).all()
    idx = O.oracle_prob_sample(p, r)
    for i in range(3):
        q = (r[i] * c[i, -1]).astype(np.float32)
        np.testing.assert_array_equal(idx[i], np.searchsorted(c[i], q, side="left").clip(0, n - 1))


def test_prob_sample_known_answer():
    # exact binary fractions: every association gives the same sums
    p = np.array([[0.5, 0.25, 0.0, 0.25, 1.0]], np.float32)
    np.testing.assert_array_equal(O.oracle_prob_cumsum(p), [[0.5, 0.75, 0.75, 1.0, 2.0]])
    r = np.array([[0.0, 0.25, 0.3, 0.375, 0.4, 0.5, 0.75, 1.0]], np.float32)
    np.testing.assert_array_equal(O.oracle_prob_sample(p, r), [[0, 0, 1, 1, 3, 3, 4, 4]])


def test_oracle_knn_composite_returns_the_k_nearest_in_order():
    """The kNN oracle (distance matrix + selection sort restatement): with distinct distances it is the plain
    ascending k-nearest list; with ties its order is whatever the selection sort's swaps produce, which is what
    the CUDA kernel is held to (tests/test_full_size_parity_gpu.py compares both with the rebuilt reference kernel)."""
    rs = np.random.RandomState(5)
    x1 = rs.random_sample((2, 60, 3)).astype(np.float32)
    x2 = rs.random_sample((2, 7, 3)).astype(np.float32)
    val, idx = O.oracle_knn_point(5, x1, x2)
    d = ((x1[:, None] - x2[:, :, None]) ** 2).sum(-1)
    order = np.argsort(d, axis=2, kind="stable")[:, :, :5]
    np.testing.assert_array_equal(idx, order.astype(np.int32))
    np.testing.assert_allclose(val, np.take_along_axis(d, order, 2), rtol=1e-6)
    # ties: 4 coincident data points -> the swap order decides; the toy case of the reference's own test
    # (test/selection_sort.cpp:68-92) is covered by the selection-sort goldens
    x1[0, 10] = x1[0, 3] = x1[0, 40] = x1[0, 0]
    val, idx = O.oracle_knn_point(6, x1, x1[:, :1].copy())
    assert sorted(idx[0, 0, :4].tolist()) == [0, 3, 10, 40] and (val[0, 0, :4] == 0).all()
