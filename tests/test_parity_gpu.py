"""GPU parity tests: the CUDA path (through the ctypes C-ABI) against
  (1) the oracle (CPU restatement) on seeded inputs,
  (2) the committed golden vectors produced by the reference's own kernels (tests/golden/),
  (3) the reference's own CUDA kernels rebuilt for sm_100a: their outputs on these tests' inputs
      (tests/golden/ref_cuda_cases.npz, a seeded sample of rows per case), and
  (4) size-independent properties at BASELINE.json's full sizes.
Bars: bit-exact for every index tensor and every copied/gathered float; three_interpolate within
1e-5 abs (it is in fact bit-exact); atomics-based gradients within 1e-4 (the reference's own bar,
tf_grouping_op_test.py:23-25)."""
import numpy as np
import pytest
import torch

from conftest import assert_golden_rows, golden_names, load_golden
from oracle import oracle as O
from pointnet2_b200 import _lib, workloads as W
from pointnet2_b200.tf_grouping import group_point, knn_point, query_ball_point, select_top_k
from pointnet2_b200.tf_interpolate import three_interpolate, three_nn, three_nn_interpolate
from pointnet2_b200.tf_sampling import farthest_point_sample, farthest_point_sample_and_gather, gather_point, prob_sample

pytestmark = pytest.mark.gpu


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def N(t):
    return t.detach().cpu().numpy()


# =============================================================================== FPS
FPS_CASES = [
    ("U", 4, 1024, 256), ("U", 2, 100, 50), ("U", 2, 40, 64), ("U", 3, 513, 100), ("D", 2, 1500, 700),
    ("S", 2, 2048, 300), ("S", 2, 3000, 128), ("U", 2, 4096, 512), ("D", 2, 5000, 200), ("U", 1, 8192, 256),
    ("U", 1, 1, 4), ("U", 2, 127, 127), ("U", 2, 129, 40), ("S", 1, 1025, 64), ("D", 2, 8192, 300), ("S", 2, 6000, 200),
    ("U", 2, 2, 5), ("U", 2, 33, 33), ("D", 3, 64, 64),
]


@pytest.mark.parametrize("gen,b,n,m", FPS_CASES)
def test_fps_matches_oracle(dev, gen, b, n, m):
    xyz = W.DISTRIBUTIONS[gen](b, n, 31)
    got = N(farthest_point_sample(m, T(xyz, dev)))
    np.testing.assert_array_equal(got, O.oracle_fps(m, xyz))


FPS_VARIANTS = [(512, 2, 2), (512, 1, 4), (512, 4, 2), (512, 8, 4), (1024, 2, 2), (512, 2, 8),
                (512, 1, 16), (512, 16, 2), (512, 32, 2), (1024, 4, 1), (512, 8, 1), (512, 16, 1),
                (256, 2, 2), (256, 8, 4), (256, 32, 2), (128, 4, 4), (128, 16, 8), (128, 32, 16), (256, 16, 16),
                (128, 2, 1), (128, 8, 1), (128, 32, 1), (256, 2, 1), (256, 4, 1), (256, 16, 1), (256, 32, 1),
                # single CTA with the chain named explicitly: cluster -1 = plain fps_step chain, -2 = packed FP32x2 chain with
                # value-only tracking (every instantiation of it)
                (128, 8, -2), (128, 16, -2), (128, 32, -2), (256, 8, -2), (256, 16, -2), (256, 32, -2), (512, 8, -2),
                (512, 16, -2), (1024, 8, -2), (128, 8, -1), (256, 16, -1), (256, 32, -1), (512, 16, -1),
                # cluster kernels with the chain named in the low bits of `threads`: +1 = packed update, +2 = plain
                (129, 4, 4), (129, 16, 8), (129, 32, 16), (257, 4, 2), (257, 8, 4), (257, 32, 2), (257, 16, 16), (513, 4, 2),
                (513, 8, 4), (513, 16, 2), (513, 32, 2), (1025, 4, 2), (1025, 8, 4), (513, 44, 2), (513, 44, 3), (513, 48, 5),
                (513, 48, 13), (513, 52, 7), (513, 52, 10), (130, 16, 8), (514, 32, 2), (514, 44, 3),
                # register + shared-memory cluster kernel (points per thread > 32), any cluster size incl. non-powers of two
                (512, 44, 2), (512, 44, 3), (512, 44, 12), (512, 44, 16), (512, 48, 5), (512, 48, 11), (512, 48, 13), (512, 52, 10), (512, 52, 7)]


@pytest.mark.parametrize("cfg", FPS_VARIANTS)
@pytest.mark.parametrize("gen", ["U", "D", "S"])
def test_fps_every_kernel_variant_matches_oracle(dev, cfg, gen):
    """Force each (threads, points/thread, cluster) kernel variant — register-resident single CTA
    (cluster 1), the DSMEM cluster exchange carrying key + coordinates (cluster >= 2) and the variant
    that streams half of the coordinates from shared memory (512 x 32) — on a cloud that fits it."""
    threads, ppt, cluster = cfg
    cap = (threads & ~3) * ppt * max(cluster, 1)
    n = min(cap, 6000) - 3
    xyz = W.DISTRIBUTIONS[gen](2, n, 32)
    lib = _lib.load()
    lib.pn2_set_fps_config(threads, ppt, cluster)
    try:
        got = N(farthest_point_sample(150, T(xyz, dev)))
    finally:
        lib.pn2_set_fps_config(0, 0, 0)
    np.testing.assert_array_equal(got, O.oracle_fps(150, xyz))


@pytest.mark.parametrize("cfg,n", [((512, 32, 16), 262144), ((512, 32, 16), 262143), ((512, 32, 2), 32768), ((256, 32, 16), 131072),
                                   ((128, 32, 16), 65536), ((256, 16, 16), 65536), ((256, 32, 8), 65536),
                                   ((512, 44, 12), 262144), ((512, 48, 11), 262144), ((512, 44, 3), 67584), ((512, 48, 7), 172032), ((512, 52, 10), 266240),
                                   # the same with the packed update (threads + 1)
                                   ((513, 32, 16), 262144), ((513, 32, 2), 32768), ((257, 32, 16), 131072), ((129, 32, 16), 65536),
                                   ((257, 16, 16), 65536), ((513, 44, 12), 262144), ((513, 48, 11), 262144), ((513, 44, 3), 67584),
                                   ((513, 52, 10), 266240)])
def test_fps_cluster_variants_at_full_capacity(dev, cfg, n):
    """The cluster kernels with EVERY per-thread slot occupied (VERDICT r1: the 512x32 variant had only
    been forced on n <= 5997, i.e. 31 of its 32 points per thread were padding).  Duplicate-heavy
    clouds so that the tie-break order crosses CTAs; checked against the oracle."""
    threads, ppt, cluster = cfg
    m = 96
    lib = _lib.load()
    for gen, b in (("U", 1), ("D", 2)):
        xyz = W.DISTRIBUTIONS[gen](b, n, 33)
        lib.pn2_set_fps_config(threads, ppt, cluster)
        try:
            fi, fx = farthest_point_sample_and_gather(m, T(xyz, dev))
        finally:
            lib.pn2_set_fps_config(0, 0, 0)
        want = O.oracle_fps(m, xyz)
        np.testing.assert_array_equal(N(fi), want)
        np.testing.assert_array_equal(N(fx), O.oracle_gather_point(xyz, want))


@pytest.mark.parametrize("chain", [-1, -2])
@pytest.mark.parametrize("gen,b,n,m,threads,ppt", [("U", 8, 4096, 1024, 256, 16), ("D", 8, 4096, 1024, 256, 16),
                                                   ("D", 4, 8192, 1024, 256, 32), ("S", 8, 2048, 700, 128, 16),
                                                   ("D", 8, 1024, 1024, 128, 8), ("D", 2, 8192, 512, 1024, 8)])
def test_fps_both_chains_match_the_reference_kernel(dev, chain, gen, b, n, m, threads, ppt):
    """The plain and the packed chain of the single-CTA kernel against the rebuilt reference kernel at the planner's
    own shapes, every per-thread slot occupied, on clouds with many exact ties (D)."""
    xyz = T(W.DISTRIBUTIONS[gen](b, n, 35), dev)
    g, case = load_golden("ref_cuda_cases"), f"fps_chains/{gen}_{b}_{n}_{m}"
    lib = _lib.load()
    lib.pn2_set_fps_config(threads, ppt, chain)
    try:
        fi, fx = farthest_point_sample_and_gather(m, xyz)
    finally:
        lib.pn2_set_fps_config(0, 0, 0)
    assert_golden_rows(fi, g, case, "idx")
    assert_golden_rows(fx, g, case, "new_xyz")


@pytest.mark.parametrize("chain", [-1, -2])
def test_fps_chains_with_ties_everywhere_and_odd_sizes(dev, chain):
    """All points coincide (every running minimum is 0 after the first pick: the tie-break alone decides every step),
    a cloud with NaN / inf coordinates, and sizes that leave padding slots in the middle of the scan order."""
    lib = _lib.load()
    rs = np.random.RandomState(36)
    clouds = [np.zeros((2, 2500, 3), np.float32) + np.float32(0.25),
              np.repeat(rs.rand(2, 7, 3).astype(np.float32), 500, axis=1)[:, :3333],
              W.cloud_uniform(2, 4093, 37), W.cloud_uniform(3, 1281, 38)]
    bad = W.cloud_uniform(2, 3000, 39)
    bad[0, 5] = np.nan
    bad[1, 77, 1] = np.inf
    bad[1, 900, 2] = -np.inf
    clouds.append(bad)
    for xyz in clouds:
        n = xyz.shape[1]
        threads, ppt = (256, 16) if n > 2048 else (128, 16)
        lib.pn2_set_fps_config(threads, ppt, chain)
        try:
            fi, fx = farthest_point_sample_and_gather(200, T(xyz, dev))
        finally:
            lib.pn2_set_fps_config(0, 0, 0)
        want = O.oracle_fps(200, xyz)
        np.testing.assert_array_equal(N(fi), want)
        np.testing.assert_array_equal(N(fx), O.oracle_gather_point(xyz, want))


def test_fps_cfg1_plumbing_matches_cpu_restatement(dev):
    """BASELINE.json configs[0]: B=8 N=1024 npoint=512 — the GPU kernels against the CPU FPS
    restatement (the reference has no CPU FPS) on the survey's input recipe."""
    c = W.CFG1_FPS_CPU
    xyz = W.cloud_uniform(c["b"], c["n"], c["seed"])
    idx = farthest_point_sample(c["npoint"], T(xyz, dev))
    assert idx.dtype == torch.int32 and tuple(idx.shape) == (8, 512)
    np.testing.assert_array_equal(N(idx), O.oracle_fps(c["npoint"], xyz))


def test_fps_tie_break_lower_slot_wins(dev):
    n = 600
    xyz = np.zeros((1, n, 3), np.float32)
    xyz[0, :, 0] = np.linspace(0.0, 0.1, n)
    xyz[0, 2] = xyz[0, 513] = (5.0, 5.0, 5.0)
    assert int(farthest_point_sample(2, T(xyz, dev))[0, 1]) == 513


@pytest.mark.parametrize("name", golden_names("fps_"))
def test_fps_and_gather_match_reference_golden(dev, name):
    g = load_golden(name)
    m = int(g["npoint"])
    idx = farthest_point_sample(m, T(g["xyz"], dev))
    np.testing.assert_array_equal(N(idx), g["idx"])
    np.testing.assert_array_equal(N(gather_point(T(g["xyz"], dev), idx)), g["new_xyz"])
    fi, fx = farthest_point_sample_and_gather(m, T(g["xyz"], dev))
    np.testing.assert_array_equal(N(fi), g["idx"])
    np.testing.assert_array_equal(N(fx), g["new_xyz"])


@pytest.mark.parametrize("gen,b,n,m", [("U", 8, 4096, 1024), ("D", 4, 8192, 1024), ("S", 32, 1024, 512),
                                       ("U", 2, 16384, 2048), ("D", 1, 65536, 1024)])
def test_fps_matches_reference_cuda_kernel(dev, gen, b, n, m):
    xyz = T(W.DISTRIBUTIONS[gen](b, n, 33), dev)
    g, case = load_golden("ref_cuda_cases"), f"fps/{gen}_{b}_{n}_{m}"
    idx = farthest_point_sample(m, xyz)
    assert_golden_rows(idx, g, case, "idx")
    fi, fx = farthest_point_sample_and_gather(m, xyz)
    assert torch.equal(fi, idx)
    assert_golden_rows(fx, g, case, "new_xyz")


def test_fps_global_scratch_fallback_matches_oracle(dev):
    """The any-size fallback (running minimum in the reference's (32,n) scratch)."""
    lib = _lib.load()
    xyz = W.cloud_uniform(3, 3000, 34)
    t = T(xyz, dev)
    out = torch.empty((3, 64), dtype=torch.int32, device=dev)
    temp = torch.empty((32, 3000), dtype=torch.float32, device=dev)
    lib.pn2_set_fps_config(1024, 0, 0)
    try:
        rc = lib.pn2_fps(3, 3000, 64, t.data_ptr(), temp.data_ptr(), out.data_ptr(), None)
    finally:
        lib.pn2_set_fps_config(0, 0, 0)
    assert rc == 0
    torch.cuda.synchronize()
    np.testing.assert_array_equal(N(out), O.oracle_fps(64, xyz))


def test_fps_full_size_properties(dev):
    """cfg2 size: indices valid, first pick 0, all picks distinct (distinct inputs), and the
    running-min distance of successive picks is non-increasing."""
    c = W.CFG2_SSG_SA
    xyz = W.cloud_uniform(c["b"], c["n"], c["seed"])
    idx = N(farthest_point_sample(c["npoint"], T(xyz, dev)))
    assert idx.shape == (c["b"], c["npoint"]) and (idx[:, 0] == 0).all()
    assert idx.min() >= 0 and idx.max() < c["n"]
    for r in idx:
        assert len(np.unique(r)) == c["npoint"]
    p = xyz[0].astype(np.float64)
    picks = p[idx[0]]
    mind = np.full(c["n"], np.inf)
    prev = np.inf
    for j in range(1, 200):
        mind = np.minimum(mind, ((p - picks[j - 1]) ** 2).sum(1))
        cur = mind[idx[0, j]]
        assert cur <= prev * (1 + 1e-6)
        assert cur >= mind.max() * (1 - 1e-5)  # it is (one of) the farthest
        prev = cur


# =============================================================================== gather_point
def test_gather_point_matches_oracle_and_grad(dev):
    xyz = W.cloud_uniform(3, 700, 35)
    idx = np.random.RandomState(36).randint(0, 700, (3, 90)).astype(np.int32)
    x = T(xyz, dev).requires_grad_(True)
    out = gather_point(x, T(idx, dev))
    np.testing.assert_array_equal(N(out), O.oracle_gather_point(xyz, idx))
    og = W.features(3, 90, 3, 37)
    out.backward(T(og, dev))
    np.testing.assert_allclose(N(x.grad), O.oracle_gather_point_grad(xyz.shape, idx, og), atol=1e-5)


# =============================================================================== ball query
BQ_CASES = [("U", 4, 1024, 128, 0.1, 32), ("U", 2, 1024, 64, 0.4, 16), ("D", 2, 2500, 96, 0.2, 32),
            ("S", 2, 700, 50, 0.2, 128), ("U", 1, 5000, 33, 0.05, 8), ("S", 3, 2049, 257, 0.3, 64),
            ("U", 2, 31, 5, 0.5, 4), ("D", 2, 4100, 10, 0.1, 1)]


@pytest.mark.parametrize("group", [0, 1, 2, 4, 8, 16, 32])
@pytest.mark.parametrize("gen,b,n,m,r,s", BQ_CASES)
def test_ball_query_matches_oracle(dev, group, gen, b, n, m, r, s):
    xyz = W.DISTRIBUTIONS[gen](b, n, 41)
    new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(m, xyz))
    _set_bq_group(group)
    try:
        idx, cnt = query_ball_point(r, s, T(xyz, dev), T(new_xyz, dev))
    finally:
        _set_bq_group(0)
    oi, oc = O.oracle_query_ball_point(r, s, xyz, new_xyz)
    np.testing.assert_array_equal(N(cnt), oc)
    np.testing.assert_array_equal(N(idx), oi)


def _set_bq_group(g):
    _lib.load().pn2_set_bq_group(g)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("gen,b,n,m,r,s", BQ_CASES + [("U", 4, 4096, 512, 0.1, 32), ("D", 3, 4096, 256, 0.1, 32), ("S", 4, 2048, 300, 0.15, 16),
                                                     ("D", 2, 8192, 200, 0.05, 8), ("U", 2, 16384, 100, 0.06, 64), ("U", 2, 300, 40, 0.02, 4)])
def test_ball_query_grid_path_matches_oracle(dev, mode, gen, b, n, m, r, s):
    """The workspace entry point against the oracle: mode 0 = automatic (shared-memory grid kernel for
    2048 <= n <= 9700, the global-memory grid beyond), mode 1 = brute force, mode 2 = the global-memory
    grid path (uniform grid for sparse balls, in-kernel ordered scan for dense ones, brute force for
    flagged clouds) at every size."""
    xyz = W.DISTRIBUTIONS[gen](b, n, 46)
    new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(m, xyz))
    lib = _lib.load()
    lib.pn2_set_bq_mode(mode)
    try:
        idx, cnt = query_ball_point(r, s, T(xyz, dev), T(new_xyz, dev))
    finally:
        lib.pn2_set_bq_mode(0)
    oi, oc = O.oracle_query_ball_point(r, s, xyz, new_xyz)
    np.testing.assert_array_equal(N(cnt), oc)
    np.testing.assert_array_equal(N(idx), oi)


@pytest.mark.parametrize("sparse_clouds", [0, 1, 2, 5, 8])
def test_ball_query_mixed_batches_follow_the_batch_rule(dev, sparse_clouds):
    """Batches mixing grid-friendly (sparse, uniform) and grid-hostile (dense surface / duplicate
    heavy) clouds: the grid serves its clouds only when >= 1/4 of the batch qualifies, otherwise
    everything goes to the brute-force kernel — either way the output is the oracle's."""
    n, m, r, s = 4096, 300, 0.08, 24
    parts = [W.cloud_uniform(1, n, 60 + i) for i in range(sparse_clouds)]
    parts += [(W.cloud_surface(1, n, 70 + i) * 0.25 if i % 2 else W.cloud_duplicates(1, n, 80 + i)) for i in range(8 - sparse_clouds)]
    xyz = np.concatenate(parts, 0).astype(np.float32)
    new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(m, xyz))
    lib = _lib.load()
    t = T(xyz, dev)
    ws_bytes = int(lib.pn2_query_ball_point_workspace_bytes(8, n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    assert lib.pn2_ball_grid_build(8, n, r, s, t.data_ptr(), ws.data_ptr(), ws_bytes, None) == 0
    torch.cuda.synchronize()
    flags = ws.view(torch.int32)[:: ws_bytes // 32][:8].cpu().numpy() != 0
    assert flags[:sparse_clouds].all() and not flags[sparse_clouds:].any(), flags
    for mode in (2, 0):
        lib.pn2_set_bq_mode(mode)
        try:
            idx, cnt = query_ball_point(r, s, t, T(new_xyz, dev))
        finally:
            lib.pn2_set_bq_mode(0)
        oi, oc = O.oracle_query_ball_point(r, s, xyz, new_xyz)
        np.testing.assert_array_equal(N(cnt), oc)
        np.testing.assert_array_equal(N(idx), oi)


def test_ball_query_grid_free_queries_outside_the_box(dev):
    """Queries outside the data's bounding box (some within the radius of border points, some far
    away) through the grid path."""
    xyz = W.cloud_uniform(2, 2000, 47)
    q = (W.cloud_uniform(2, 300, 48) * 1.5 - 0.25).astype(np.float32)
    q[:, :20] += 5.0
    idx, cnt = query_ball_point(0.08, 16, T(xyz, dev), T(q, dev))
    oi, oc = O.oracle_query_ball_point(0.08, 16, xyz, q)
    np.testing.assert_array_equal(N(cnt), oc)
    np.testing.assert_array_equal(N(idx), oi)
    assert (oc == 0).any() and (oc > 0).any()


def test_ball_query_free_queries_and_empty_rows(dev):
    """Queries that are not data points: empty balls give zero rows and pts_cnt 0."""
    xyz = W.cloud_uniform(2, 300, 42)
    q = (W.cloud_uniform(2, 40, 43) * 1.6 - 0.3).astype(np.float32)
    idx, cnt = query_ball_point(0.15, 8, T(xyz, dev), T(q, dev))
    oi, oc = O.oracle_query_ball_point(0.15, 8, xyz, q)
    np.testing.assert_array_equal(N(idx), oi)
    np.testing.assert_array_equal(N(cnt), oc)
    assert (oc == 0).any() and (N(idx)[oc == 0] == 0).all()


def test_ball_query_boundary_ulps(dev):
    """Points placed within a few ulps of the radius on both sides: the sqrt-free threshold
    must agree with the reference's max(sqrtf(d2),1e-20f) < radius test."""
    rs = np.random.RandomState(44)
    r = np.float32(0.2)
    n = 4096
    dirs = rs.normal(size=(n, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    scale = r * (1.0 + rs.randint(-6, 7, n) * 2.0 ** -24)
    xyz = (dirs * scale[:, None]).astype(np.float32)[None]
    q = np.zeros((1, 1, 3), np.float32)
    idx, cnt = query_ball_point(float(r), 4096, T(xyz, dev), T(q, dev))
    oi, oc = O.oracle_query_ball_point(float(r), 4096, xyz, q)
    assert 0 < int(oc[0, 0]) < n
    np.testing.assert_array_equal(N(cnt), oc)
    np.testing.assert_array_equal(N(idx), oi)


def test_ball_threshold_matches_oracle():
    lib = _lib.load()
    for r in [0.1, 0.2, 0.4, 0.8, 0.05, 1e-3, 3.0, 1e-19, 1e-20, 1e-21, 1e30]:
        assert float(lib.pn2_ball_threshold(r)) == O.oracle_ball_threshold(r)


@pytest.mark.parametrize("name", golden_names("bq_"))
def test_ball_query_and_group_match_reference_golden(dev, name):
    g = load_golden(name)
    idx, cnt = query_ball_point(float(g["radius"]), int(g["nsample"]), T(g["xyz"], dev), T(g["new_xyz"], dev))
    np.testing.assert_array_equal(N(cnt), g["pts_cnt"])
    np.testing.assert_array_equal(N(idx), g["idx"])
    if "grouped_xyz" in g:
        np.testing.assert_array_equal(N(group_point(T(g["xyz"], dev), idx)), g["grouped_xyz"])
        np.testing.assert_array_equal(N(group_point(T(g["feats"], dev), idx)), g["grouped_feats"])


@pytest.mark.parametrize("gen,b,n,m,r,s", [("U", 8, 4096, 1024, 0.1, 32), ("D", 4, 8192, 1024, 0.1, 32),
                                           ("S", 8, 1024, 512, 0.4, 128), ("S", 8, 512, 128, 0.8, 128)])
def test_ball_query_and_group_match_reference_cuda_kernel(dev, gen, b, n, m, r, s):
    xyz = T(W.DISTRIBUTIONS[gen](b, n, 45), dev)
    g, case = load_golden("ref_cuda_cases"), f"bq/{gen}_{b}_{n}_{m}_{r}_{s}"
    _, new_xyz = farthest_point_sample_and_gather(m, xyz)  # the reference's centroids (checked below)
    assert_golden_rows(new_xyz, g, case, "new_xyz")
    idx, cnt = query_ball_point(r, s, xyz, new_xyz)
    assert_golden_rows(cnt, g, case, "cnt")
    assert_golden_rows(idx, g, case, "idx")
    grouped = group_point(xyz, idx)
    assert_golden_rows(grouped, g, case, "grouped")
    np.testing.assert_array_equal(N(grouped), O.oracle_group_point(N(xyz), N(idx)))


def test_ball_query_full_size_properties(dev):
    c = W.CFG2_SSG_SA
    xyz = W.cloud_uniform(c["b"], c["n"], c["seed"])
    x = T(xyz, dev)
    fi, new_xyz = farthest_point_sample_and_gather(c["npoint"], x)
    idx, cnt = query_ball_point(c["radius"], c["nsample"], x, new_xyz)
    idx, cnt, nx = N(idx), N(cnt), N(new_xyz)
    assert idx.min() >= 0 and idx.max() < c["n"] and cnt.min() >= 1 and cnt.max() <= c["nsample"]
    b0 = 0
    d = np.sqrt(((xyz[b0][idx[b0]].astype(np.float64) - nx[b0][:, None, :]) ** 2).sum(-1))
    assert (d < c["radius"] + 1e-6).all()  # every returned index is inside the ball
    for j in range(0, c["npoint"], 37):  # real hits ascending, padding equals the first hit
        k = cnt[b0, j]
        assert (np.diff(idx[b0, j, :k]) > 0).all()
        assert (idx[b0, j, k:] == idx[b0, j, 0]).all()
    # idempotence of the count: exact recount of one row in float64 away from the boundary
    dd = np.sqrt(((xyz[b0].astype(np.float64) - nx[b0][5]) ** 2).sum(-1))
    assert min(int((dd < c["radius"] - 1e-6).sum()), c["nsample"]) <= cnt[b0, 5] <= int((dd < c["radius"] + 1e-6).sum())


# =============================================================================== group_point
@pytest.mark.parametrize("c", [3, 1, 4, 16, 64, 67, 320, 5])
def test_group_point_matches_oracle(dev, c):
    rs = np.random.RandomState(51)
    pts = W.features(3, 333, c, 52)
    idx = rs.randint(0, 333, (3, 37, 9)).astype(np.int32)
    np.testing.assert_array_equal(N(group_point(T(pts, dev), T(idx, dev))), O.oracle_group_point(pts, idx))


@pytest.mark.parametrize("c", [3, 16, 7])
def test_group_point_grad_matches_oracle(dev, c):
    rs = np.random.RandomState(53)
    pts = W.features(2, 200, c, 54)
    idx = rs.randint(0, 200, (2, 30, 8)).astype(np.int32)
    p = T(pts, dev).requires_grad_(True)
    out = group_point(p, T(idx, dev))
    go = W.features(2, 30 * 8, c, 55).reshape(2, 30, 8, c)
    out.backward(T(go, dev))
    np.testing.assert_allclose(N(p.grad), O.oracle_group_point_grad(pts.shape, idx, go), atol=1e-4, rtol=1e-5)


def test_group_point_gradient_error_like_reference_test(dev):
    """tf_ops/grouping/tf_grouping_op_test.py:9-25: numerical vs analytical gradient of
    group_point(points, query_ball_point(0.3, 32, xyz1, xyz2)) on (1,128,16)/(1,8,3), < 1e-4."""
    rs = np.random.RandomState(56)
    points = rs.random_sample((1, 128, 16)).astype(np.float32)
    xyz1 = rs.random_sample((1, 128, 3)).astype(np.float32)
    xyz2 = rs.random_sample((1, 8, 3)).astype(np.float32)
    idx, _ = query_ball_point(0.3, 32, T(xyz1, dev), T(xyz2, dev))
    p = T(points, dev).requires_grad_(True)
    w = T(rs.standard_normal((1, 8, 32, 16)).astype(np.float32), dev)
    (group_point(p, idx) * w).sum().backward()
    analytic = N(p.grad)
    i = N(idx)
    num = np.zeros_like(points, dtype=np.float64)
    np.add.at(num[0], i[0].reshape(-1), N(w)[0].reshape(-1, 16).astype(np.float64))  # d(sum w*out)/dpoints, linear op
    assert np.abs(analytic - num).max() < 1e-4


def test_group_point_full_size_linearity(dev):
    """cfg3 layer-2 size (C=320, S=128): group(a*p + q) == a*group(p) + group(q) exactly for a
    power-of-two a (pure copies), and a checksum of the output equals the checksum predicted from
    the index histogram."""
    rs = np.random.RandomState(57)
    b, n, c, m, s = 4, 512, 320, 128, 128
    p = T(W.features(b, n, c, 58), dev)
    q = T(W.features(b, n, c, 59), dev)
    idx = T(rs.randint(0, n, (b, m, s)).astype(np.int32), dev)
    gp, gq = group_point(p, idx), group_point(q, idx)
    assert torch.equal(group_point(2.0 * p + q, idx), (2.0 * p + q).gather(1, idx.long().reshape(b, -1, 1).expand(-1, -1, c)).reshape(b, m, s, c))
    assert torch.equal(gp, p.gather(1, idx.long().reshape(b, -1, 1).expand(-1, -1, c)).reshape(b, m, s, c))
    hist = torch.zeros((b, n), dtype=torch.float64, device=dev)
    hist.scatter_add_(1, idx.long().reshape(b, -1), torch.ones((b, m * s), dtype=torch.float64, device=dev))
    want = (hist.unsqueeze(-1) * q.double()).sum()
    assert abs(float(gq.double().sum() - want)) < 1e-6 * max(1.0, abs(float(want)))


# =============================================================================== three_nn / interpolate
@pytest.mark.parametrize("n,m,dup", [(600, 150, False), (400, 100, True), (30, 2, False), (10, 1, False),
                                     (2500, 2100, False), (129, 4, True), (1, 3, False)])
def test_three_nn_matches_oracle(dev, n, m, dup):
    xyz1 = W.cloud_duplicates(2, n, 61, drop=False) if dup else W.cloud_uniform(2, n, 61)
    xyz2 = xyz1[:, :m].copy() if dup else W.cloud_uniform(2, m, 62)
    d, i = three_nn(T(xyz1, dev), T(xyz2, dev))
    od, oi = O.oracle_three_nn(xyz1, xyz2)
    np.testing.assert_array_equal(N(i), oi)
    np.testing.assert_array_equal(N(d), od)


@pytest.mark.parametrize("c", [64, 5, 128, 1])
def test_three_interpolate_matches_oracle_and_grad(dev, c):
    xyz1, xyz2 = W.cloud_uniform(2, 300, 63), W.cloud_uniform(2, 60, 64)
    pts = W.features(2, 60, c, 65)
    d, i = O.oracle_three_nn(xyz1, xyz2)
    dd = np.maximum(d, 1e-10)
    w = ((1.0 / dd) / (1.0 / dd).sum(axis=2, keepdims=True)).astype(np.float32)
    p = T(pts, dev).requires_grad_(True)
    out = three_interpolate(p, T(i, dev), T(w, dev))
    want = O.oracle_three_interpolate(pts, i, w)
    assert np.abs(N(out) - want).max() <= 1e-5  # the contract
    np.testing.assert_array_equal(N(out), want)  # and in fact bit-exact
    go = W.features(2, 300, c, 66)
    out.backward(T(go, dev))
    np.testing.assert_allclose(N(p.grad), O.oracle_three_interpolate_grad(pts.shape, i, w, go), atol=1e-4, rtol=1e-5)


@pytest.mark.parametrize("name", golden_names("interp_"))
def test_interpolation_matches_reference_golden(dev, name):
    g = load_golden(name)
    d, i = three_nn(T(g["xyz1"], dev), T(g["xyz2"], dev))
    np.testing.assert_array_equal(N(i), g["idx"])
    np.testing.assert_array_equal(N(d), g["dist"])
    p = T(g["points"], dev).requires_grad_(True)
    out = three_interpolate(p, i, T(g["weight"], dev))
    assert np.abs(N(out) - g["out"]).max() <= 1e-5
    out.backward(T(g["grad_out"], dev))
    np.testing.assert_allclose(N(p.grad), g["grad_points"], atol=1e-4, rtol=1e-5)


def test_three_interpolate_gradient_error_like_reference_test(dev):
    """tf_ops/3d_interpolation/tf_interpolate_op_test.py:9-21: constant 1/3 weights,
    (1,8,16) -> (1,128,16), gradient error < 1e-4."""
    rs = np.random.RandomState(67)
    points = rs.random_sample((1, 8, 16)).astype(np.float32)
    xyz1 = rs.random_sample((1, 128, 3)).astype(np.float32)
    xyz2 = rs.random_sample((1, 8, 3)).astype(np.float32)
    _, idx = three_nn(T(xyz1, dev), T(xyz2, dev))
    weight = torch.full((1, 128, 3), 1.0 / 3.0, dtype=torch.float32, device=dev)
    p = T(points, dev).requires_grad_(True)
    g = T(rs.standard_normal((1, 128, 16)).astype(np.float32), dev)
    (three_interpolate(p, idx, weight) * g).sum().backward()
    num = np.zeros((8, 16))
    i = N(idx)[0]
    for t in range(3):
        np.add.at(num, i[:, t], N(g)[0].astype(np.float64) / 3.0)
    assert np.abs(N(p.grad)[0] - num).max() < 1e-4


@pytest.mark.parametrize("n,m,c", [(500, 120, 64), (77, 9, 5), (64, 16, 512), (300, 2, 8)])
def test_fused_three_nn_interpolate_matches_unfused(dev, n, m, c):
    xyz1, xyz2 = W.cloud_uniform(2, n, 68), W.cloud_uniform(2, m, 69)
    pts = W.features(2, m, c, 70)
    out, d, i, w = three_nn_interpolate(T(xyz1, dev), T(xyz2, dev), T(pts, dev), return_aux=True)
    od, oi = O.oracle_three_nn(xyz1, xyz2)
    np.testing.assert_array_equal(N(i), oi)
    np.testing.assert_array_equal(N(d), od)
    dd = np.maximum(od, np.float32(1e-10))
    r = (np.float32(1.0) / dd).astype(np.float32)
    norm = ((r[..., 0] + r[..., 1]) + r[..., 2]).astype(np.float32)
    ww = (r / norm[..., None]).astype(np.float32)
    np.testing.assert_allclose(N(w), ww, rtol=2e-7, atol=0)
    want = O.oracle_three_interpolate(pts, oi, N(w))
    np.testing.assert_array_equal(N(out), want)
    assert np.abs(N(three_nn_interpolate(T(xyz1, dev), T(xyz2, dev), T(pts, dev))) - want).max() <= 1e-5


def test_fp_stack_full_size_roundtrip(dev):
    """cfg4 last FP layer size (16 x 8192 <- 1024, C=128): interpolating a LINEAR field sampled at
    the known points reproduces it at every unknown point that coincides with a known point
    (weight ~1 on the zero-distance neighbour), and stays inside the convex hull elsewhere."""
    b, n, m, c = 16, 8192, 1024, 128
    xyz1 = W.cloud_uniform(b, n, 71)
    x1 = T(xyz1, dev)
    x2 = x1[:, :m].contiguous()
    A = T(np.random.RandomState(72).standard_normal((3, c)).astype(np.float32), dev)
    f2 = x2 @ A
    out, d, i, w = three_nn_interpolate(x1, x2, f2, return_aux=True)
    assert torch.equal(i[:, :m, 0], torch.arange(m, device=dev, dtype=torch.int32).expand(b, m))
    assert float(d[:, :m, 0].abs().max()) == 0.0
    assert float((out[:, :m] - f2).abs().max()) < 1e-4
    lo = torch.minimum(torch.minimum(f2.gather(1, i[..., 0].long().unsqueeze(-1).expand(-1, -1, c)),
                                     f2.gather(1, i[..., 1].long().unsqueeze(-1).expand(-1, -1, c))),
                       f2.gather(1, i[..., 2].long().unsqueeze(-1).expand(-1, -1, c)))
    assert bool((out >= lo - 1e-4).all())
    assert float((w.sum(-1) - 1).abs().max()) < 1e-5


# =============================================================================== selection sort / knn
def test_select_top_k_matches_oracle_and_golden(dev):
    dist = np.random.RandomState(81).random_sample((2, 6, 40)).astype(np.float32)
    dist[0, 0, 5] = dist[0, 0, 17]
    oi, ov = select_top_k(7, T(dist, dev))
    ri, rv = O.oracle_selection_sort(7, dist)
    np.testing.assert_array_equal(N(oi), ri)
    np.testing.assert_array_equal(N(ov), rv)
    for name in golden_names("selection_sort"):
        g = load_golden(name)
        gi, gv = select_top_k(int(g["k"]), T(g["dist"], dev))
        np.testing.assert_array_equal(N(gi), g["outi"])
        np.testing.assert_array_equal(N(gv), g["out"])


def test_knn_point_returns_k_nearest(dev):
    xyz1, xyz2 = W.cloud_uniform(2, 200, 82), W.cloud_uniform(2, 30, 83)
    val, idx = knn_point(5, T(xyz1, dev), T(xyz2, dev))
    d = ((xyz1[:, None, :, :] - xyz2[:, :, None, :]) ** 2).sum(-1)
    np.testing.assert_allclose(N(val), np.sort(d, axis=2)[:, :, :5], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(np.take_along_axis(d, N(idx).astype(np.int64), 2), N(val), rtol=1e-5, atol=1e-7)


# =============================================================================== launches really happen on the device
def test_kernels_launch_and_library_is_in_tree(dev):
    import os
    before = _lib.launch_count()
    xyz = T(W.cloud_uniform(1, 64, 91), dev)
    farthest_point_sample(4, xyz)
    assert _lib.launch_count() == before + 1
    assert os.path.dirname(_lib.lib_path()).endswith("pointnet2_b200")


# ------------------------------------------------------------------------------- prob_sample
@pytest.mark.parametrize("b,n,m", [(1, 1, 5), (3, 5, 64), (4, 1000, 300), (2, 8192, 100), (2, 8193, 100), (3, 30000, 1000),
                                   (40, 257, 33)])
def test_prob_sample_matches_oracle(dev, b, n, m):
    rng = np.random.RandomState(n + m)
    p = rng.random_sample((b, n)).astype(np.float32)
    if n > 100:
        p[:, rng.randint(0, n, n // 3)] = 0.0
    r = rng.random_sample((b, m)).astype(np.float32)
    r[:, 0] = 0.0
    r[:, -1] = 1.0
    np.testing.assert_array_equal(N(prob_sample(T(p, dev), T(r, dev))), O.oracle_prob_sample(p, r))


@pytest.mark.parametrize("name", golden_names("prob_"))
def test_prob_sample_matches_reference_golden(dev, name):
    g = load_golden(name)
    np.testing.assert_array_equal(N(prob_sample(T(g["inp"], dev), T(g["inpr"], dev))), g["out"])
    lib = _lib.load()
    p = T(g["inp"], dev)
    temp = torch.empty_like(p)
    assert lib.pn2_prob_sample(p.shape[0], p.shape[1], 0, p.data_ptr(), None, temp.data_ptr(), None, None) == 0
    torch.cuda.synchronize()
    np.testing.assert_array_equal(N(temp), g["cumsum"])  # the scratch holds the reference's cumulative sums


@pytest.mark.parametrize("b,n,m", [(8, 4096, 2048), (2, 100000, 4096), (33, 777, 100)])
def test_prob_sample_matches_reference_cuda_kernel(dev, b, n, m):
    rng = np.random.RandomState(b + n)
    p = rng.random_sample((b, n)).astype(np.float32)
    r = rng.random_sample((b, m)).astype(np.float32)
    out = N(prob_sample(T(p, dev), T(r, dev)))
    assert_golden_rows(out, load_golden("ref_cuda_cases"), f"prob/{b}_{n}_{m}", "out")
    np.testing.assert_array_equal(out, O.oracle_prob_sample(p, r))


def test_prob_sample_rejects_bad_shapes(dev):
    with pytest.raises(ValueError):
        prob_sample(torch.zeros(4, device=dev), torch.zeros(1, 4, device=dev))
    with pytest.raises(ValueError):
        prob_sample(torch.zeros(2, 4, device=dev), torch.zeros(3, 4, device=dev))
    with pytest.raises(TypeError):
        prob_sample(torch.zeros(2, 4, device=dev, dtype=torch.float64), torch.zeros(2, 4, device=dev))


@pytest.mark.parametrize("n", [131073, 262144, 262145, 300001])
def test_fps_at_and_beyond_the_cluster_capacity(dev, n):
    """The planner's last two regimes as the planner picks them (no forced config): 16-CTA clusters
    with coordinates in shared memory up to n = 262144, the global-scratch fallback beyond."""
    xyz = W.cloud_uniform(2, n, 91)
    want = O.oracle_fps(6, xyz)
    t = T(xyz, dev)
    np.testing.assert_array_equal(N(farthest_point_sample(6, t)), want)
    fi, fx = farthest_point_sample_and_gather(6, t)
    np.testing.assert_array_equal(N(fi), want)
    np.testing.assert_array_equal(N(fx), O.oracle_gather_point(xyz, want))


@pytest.mark.parametrize("n", [600, 5000])
def test_ball_query_non_finite_points_follow_the_reference(dev, n):
    """A NaN point is a hit in every ball, an infinite one in none (tf_grouping_g.cu:24-25 with
    fmaxf): the uniform-grid path must step aside for such clouds and the scan must agree with
    the oracle."""
    xyz = W.cloud_uniform(3, n, 95)
    xyz[0, 17] = np.nan
    xyz[0, n // 2, 1] = np.nan
    xyz[1, 40, 2] = np.inf
    q = O.oracle_gather_point(xyz[:, ::3].copy(), O.oracle_fps(64, xyz[:, ::3].copy()))
    q[~np.isfinite(q)] = 0.5
    idx, cnt = query_ball_point(0.06, 16, T(xyz, dev), T(q, dev))
    oi, oc = O.oracle_query_ball_point(0.06, 16, xyz, q)
    np.testing.assert_array_equal(N(cnt), oc)
    np.testing.assert_array_equal(N(idx), oi)
    assert (oi[0] == 17).any()
