"""Generate golden vectors for tests/golden/ from the REFERENCE'S OWN code (TEST INFRASTRUCTURE).

Runs on a GPU box (the reference's sampling/grouping ops are GPU-only, tf_sampling.cpp:123,
tf_grouping.cpp:106): executes the reference CUDA kernels rebuilt unmodified for sm_100a
(oracle/_ref/libref_{sampling,grouping}.so) and the reference CPU functions
(oracle/_ref/libref_cpu.so) on small seeded inputs and stores inputs + outputs as .npz.

    python oracle/gen_golden.py OUTDIR                  # on a GPU machine, after oracle/build.py
    python oracle/gen_golden.py --ref-cases-cpu OUTDIR  # ref_cpu_cases.npz, no GPU needed
    python oracle/gen_golden.py --ref-cases-gpu OUTDIR  # ref_cuda_cases.npz, on a GPU machine
    cp OUTDIR/*.npz tests/golden/

The fixtures pin the oracle (tests/test_oracle_golden.py, CPU) and the CUDA path
(tests/test_parity_gpu.py, GPU).  ref_{cpu,cuda}_cases.npz hold the reference's outputs on the
very inputs of the tests that compare with the reference's own code, so those tests run where the
reference is not built.  Per output: ``<case>/<output>.shape`` and ``<case>/<output>.sha256`` (of the
whole output's bytes), and rows over the two leading axes, ``<case>/<output>`` at the row numbers
``<case>/pos`` (every row of the small outputs, a seeded sample of the large ones), so that a
mismatch shows where it is; see tests/conftest.py:assert_golden_rows.
"""
from __future__ import annotations

import hashlib
import os
import sys
import zipfile
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import oracle as O  # noqa: E402
from pointnet2_b200 import workloads as W  # noqa: E402


def prob_cases():
    """ProbSample inputs: (probabilities (b,n), uniform draws (b,m))."""
    rng = np.random.RandomState(150)
    cases = {}
    for name, n, m in (("prob_n5", 5, 64), ("prob_n1000", 1000, 256), ("prob_two_chunks", 9000, 256)):
        p = rng.random_sample((2, n)).astype(np.float32)
        if n >= 1000:
            p[:, rng.randint(0, n, n // 3)] = 0.0  # plateaus in the cumulative sum
        r = rng.random_sample((2, m)).astype(np.float32)
        r[:, 0], r[:, 1] = 0.0, 1.0
        cases[name] = (p, r)
    return cases


def main_prob(outdir: str) -> None:
    """Only the ProbSample fixtures (added after the first fixture set was committed)."""
    import torch
    assert torch.cuda.is_available()
    dev = torch.device("cuda:0")
    os.makedirs(outdir, exist_ok=True)
    for name, (p, r) in prob_cases().items():
        out, cum = O.refcuda_prob_sample(torch.from_numpy(p).to(dev), torch.from_numpy(r).to(dev), return_cumsum=True)
        np.savez_compressed(os.path.join(outdir, name + ".npz"), inp=p, inpr=r, cumsum=cum.cpu().numpy(), out=out.cpu().numpy())
        print("wrote", name)


def main(outdir: str) -> None:
    import torch
    assert torch.cuda.is_available(), "gen_golden.py needs a GPU: the reference's FPS/ball-query kernels are GPU-only"
    dev = torch.device("cuda:0")
    os.makedirs(outdir, exist_ok=True)

    def t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    def save(name, **arrs):
        savez_lzma(os.path.join(outdir, name + ".npz"), arrs)
        print("wrote", name, {k: v.shape for k, v in arrs.items()})

    # ---- FPS + gather_point (reference CUDA) --------------------------------------------------
    fps_cases = {
        "fps_uniform": (W.cloud_uniform(4, 1024, 100), 256),      # cfg1-like
        "fps_dups": (W.cloud_duplicates(2, 1500, 101), 700),      # real ties; npoint > #distinct
        "fps_small_n": (W.cloud_uniform(3, 100, 102), 50),        # n < 512: empty slots
        "fps_beyond_smem": (W.cloud_surface(2, 5000, 103), 64),   # n > 3072: reference's global path
        "fps_npoint_gt_n": (W.cloud_uniform(2, 40, 104), 64),     # npoint > n
    }
    for name, (xyz, m) in fps_cases.items():
        idx = O.refcuda_fps(m, t(xyz))
        new_xyz = O.refcuda_gather_point(t(xyz), idx)
        save(name, xyz=xyz, npoint=np.int32(m), idx=idx.cpu().numpy(), new_xyz=new_xyz.cpu().numpy())

    # ---- ball query + group_point (reference CUDA) -------------------------------------------
    bq_cases = {
        "bq_uniform_r0.1": (W.cloud_uniform(4, 1024, 110), 128, 0.1, 32),   # sparse: rows padded
        "bq_uniform_r0.4": (W.cloud_uniform(2, 1024, 111), 64, 0.4, 16),    # dense: early exit
        "bq_dups_r0.2": (W.cloud_duplicates(2, 2500, 112), 96, 0.2, 32),    # coincident points, tile boundary
        "bq_surface_r0.2_s128": (W.cloud_surface(2, 700, 113), 50, 0.2, 128),
    }
    for name, (xyz, m, r, s) in bq_cases.items():
        fidx = O.refcuda_fps(m, t(xyz))
        new_xyz = O.refcuda_gather_point(t(xyz), fidx)
        idx, cnt = O.refcuda_query_ball_point(r, s, t(xyz), new_xyz)
        grouped = O.refcuda_group_point(t(xyz), idx)
        feats = W.features(xyz.shape[0], xyz.shape[1], 16, 7)
        gfeat = O.refcuda_group_point(t(feats), idx)
        save(name, xyz=xyz, new_xyz=new_xyz.cpu().numpy(), radius=np.float32(r), nsample=np.int32(s),
             idx=idx.cpu().numpy(), pts_cnt=cnt.cpu().numpy(), grouped_xyz=grouped.cpu().numpy(),
             feats=feats, grouped_feats=gfeat.cpu().numpy())
    # queries that are NOT data points and may have empty balls (rows left to the pre-zeroed buffer)
    xyz = W.cloud_uniform(2, 300, 114)
    q = (W.cloud_uniform(2, 40, 115) * 1.6 - 0.3).astype(np.float32)
    idx, cnt = O.refcuda_query_ball_point(0.15, 8, t(xyz), t(q))
    save("bq_free_queries", xyz=xyz, new_xyz=q, radius=np.float32(0.15), nsample=np.int32(8),
         idx=idx.cpu().numpy(), pts_cnt=cnt.cpu().numpy())

    # ---- selection sort (reference CUDA) -----------------------------------------------------
    dist = np.random.RandomState(120).random_sample((2, 6, 40)).astype(np.float32)
    dist[0, 0, 5] = dist[0, 0, 17]  # a tie
    outi, out = O.refcuda_selection_sort(7, t(dist))
    save("selection_sort", dist=dist, k=np.int32(7), outi=outi.cpu().numpy(), out=out.cpu().numpy())
    # the reference's only known-answer case (test/selection_sort.cpp:68-92): dist = 10 - i
    kat = np.tile((10.0 - np.arange(4, dtype=np.float32)), (2, 2, 1))
    outi, out = O.refcuda_selection_sort(3, t(kat))
    save("selection_sort_kat", dist=kat, k=np.int32(3), outi=outi.cpu().numpy(), out=out.cpu().numpy())

    # ---- three_nn / three_interpolate (reference CPU) -----------------------------------------
    for name, (n, m, c, seed) in {"interp_1024_256_c64": (1024, 256, 64, 130), "interp_64_16_c5": (64, 16, 5, 131),
                                  "interp_m2": (20, 2, 8, 132)}.items():
        xyz1 = W.cloud_duplicates(2, n, seed, drop=False) if "1024" in name else W.cloud_uniform(2, n, seed)
        xyz2 = xyz1[:, :m].copy() if "1024" in name else W.cloud_uniform(2, m, seed + 1)
        pts = W.features(2, m, c, seed + 2)
        d, i = O.refcpu_three_nn(xyz1, xyz2)
        dd = np.maximum(d, 1e-10)
        w = ((1.0 / dd) / (1.0 / dd).sum(axis=2, keepdims=True)).astype(np.float32)
        w = np.nan_to_num(w, nan=0.0, posinf=0.0, neginf=0.0).astype(np.float32)
        out = O.refcpu_three_interpolate(pts, i, w)
        go = W.features(2, n, c, seed + 3)
        gp = O.refcpu_three_interpolate_grad(pts.shape, i, w, go)
        save(name, xyz1=xyz1, xyz2=xyz2, points=pts, dist=d, idx=i, weight=w, out=out, grad_out=go, grad_points=gp)

    # ---- gradients of gather/group (reference CUDA, float atomics: compare with tolerance) ----
    xyz = W.cloud_uniform(2, 256, 140)
    fidx = O.refcuda_fps(32, t(xyz))
    new_xyz = O.refcuda_gather_point(t(xyz), fidx)
    idx, _ = O.refcuda_query_ball_point(0.3, 16, t(xyz), new_xyz)
    feats = W.features(2, 256, 12, 141)
    go = W.features(2, 32 * 16, 12, 142).reshape(2, 32, 16, 12)
    gp = O.refcuda_group_point_grad(feats.shape, idx, t(go))
    og = W.features(2, 32, 3, 143)
    gi = O.refcuda_gather_point_grad(xyz.shape, fidx, t(og))
    save("grads", xyz=xyz, fps_idx=fidx.cpu().numpy(), idx=idx.cpu().numpy(), feats=feats, grad_out=go,
         grad_points=gp.cpu().numpy(), out_g=og, inp_g=gi.cpu().numpy())
    main_prob(outdir)
    print("golden vectors written to", outdir)


def savez_lzma(path: str, arrays: dict) -> None:
    """np.savez with LZMA members (np.load reads them): keeps the larger fixtures under 1 MB."""
    import io
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for k, v in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asarray(v), allow_pickle=False)
            z.writestr(k + ".npy", buf.getvalue())


class _Rows(dict):
    """Collects, for each output of a case, its shape and the sha256 of its bytes (the whole output), and a
    seeded sample of its rows over the two leading axes (all rows when ``k`` is None) for readable failures."""

    def add(self, case: str, k: int | None, **outs) -> None:
        a0 = np.asarray(next(iter(outs.values())))
        nrows = a0.shape[0] * a0.shape[1]
        pos = np.arange(nrows) if k is None or k >= nrows else \
            np.sort(np.random.RandomState(zlib.crc32(case.encode())).choice(nrows, k, replace=False))
        self[case + "/pos"] = pos.astype(np.int32)
        for name, a in outs.items():
            a = np.ascontiguousarray(a)
            assert a.shape[0] * a.shape[1] == nrows
            self[case + "/" + name] = a.reshape(nrows, -1)[pos]
            self[case + "/" + name + ".shape"] = np.array(a.shape, np.int64)
            self[case + "/" + name + ".sha256"] = np.array(hashlib.sha256(a.tobytes()).hexdigest())


def main_ref_cases_cpu(outdir: str) -> None:
    """The reference's CPU functions on the inputs of test_oracle_cpu.py and of
    test_fp_and_concat_gpu.py's deterministic three_interpolate gradient cases."""
    rows = _Rows()
    for r, s in ((0.1, 32), (0.4, 16), (0.05, 8)):
        xyz = W.cloud_uniform(3, 800, 11)
        new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(100, xyz))
        rows.add(f"bq_nofma/{r}_{s}", None, idx=O.refcpu_query_ball_point(r, s, xyz, new_xyz))
    xyz = W.cloud_uniform(2, 500, 12)
    feats = W.features(2, 500, 7, 13)
    new_xyz = O.oracle_gather_point(xyz, O.oracle_fps(64, xyz))
    idx, _ = O.oracle_query_ball_point(0.2, 16, xyz, new_xyz)
    rows.add("group", None, out=O.refcpu_group_point(feats, idx))
    go = W.features(2, 64 * 16, 7, 14).reshape(2, 64, 16, 7)
    rows.add("group_grad", None, out=O.refcpu_group_point_grad(feats.shape, idx, go))
    for n, m, dup in ((600, 150, False), (400, 100, True), (30, 2, False), (10, 1, False)):
        xyz1 = W.cloud_duplicates(2, n, 15, drop=False) if dup else W.cloud_uniform(2, n, 15)
        xyz2 = xyz1[:, :m].copy() if dup else W.cloud_uniform(2, m, 16)
        rd, ri = O.refcpu_three_nn(xyz1, xyz2)
        rows.add(f"three_nn/{n}_{m}_{dup}", None, dist=rd, idx=ri)
    xyz1, xyz2 = W.cloud_uniform(2, 300, 17), W.cloud_uniform(2, 60, 18)
    pts = W.features(2, 60, 33, 19)
    d, i = O.oracle_three_nn(xyz1, xyz2)
    dd = np.maximum(d, 1e-10)
    w = ((1.0 / dd) / (1.0 / dd).sum(axis=2, keepdims=True)).astype(np.float32)
    rows.add("three_interp", None, out=O.refcpu_three_interpolate(pts, i, w))
    go = W.features(2, 300, 33, 20)
    rows.add("three_interp_grad", None, out=O.refcpu_three_interpolate_grad(pts.shape, i, w, go))
    for b, n, m, c in ((16, 8192, 1024, 128), (4, 1024, 256, 256), (2, 300, 40, 7), (2, 64, 16, 512), (3, 500, 1, 8),
                       (2, 500, 2, 33), (1, 20000, 5, 16), (2, 10, 300, 4), (2, 3000, 60, 132)):
        x1, x2 = W.cloud_uniform(b, n, 211), W.cloud_uniform(b, m, 212)
        _, idx = O.oracle_three_nn(x1, x2)
        w = np.random.RandomState(213).random_sample((b, n, 3)).astype(np.float32)
        go = W.features(b, n, c, 214)
        rows.add(f"three_interp_grad_det/{b}_{n}_{m}_{c}", 8, out=O.refcpu_three_interpolate_grad((b, m, c), idx, w, go))
    os.makedirs(outdir, exist_ok=True)
    savez_lzma(os.path.join(outdir, "ref_cpu_cases.npz"), rows)
    print("wrote ref_cpu_cases", len(rows), "arrays")


def main_ref_cases_gpu(outdir: str) -> None:
    """The reference's CUDA kernels (and, for the FP stack, its CPU functions) on the inputs of the
    tests in test_parity_gpu.py and test_full_size_parity_gpu.py that compare with them; inputs
    that the tests derive with this library's own ops are derived the same way here."""
    import torch

    from pointnet2_b200.tf_interpolate import three_nn
    from pointnet2_b200.tf_sampling import farthest_point_sample, farthest_point_sample_and_gather, gather_point
    assert torch.cuda.is_available() and O.have_refcuda(), "needs a GPU and oracle/_ref (oracle/build.py)"
    dev = torch.device("cuda:0")
    rows = _Rows()
    rows["meta/device"] = np.array(torch.cuda.get_device_name(dev))

    def t(a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    def n_(x):
        return x.cpu().numpy()

    def fps(key, x, m, k):
        ref = O.refcuda_fps(m, x)
        rows.add(key, k, idx=n_(ref), new_xyz=n_(O.refcuda_gather_point(x, ref)))

    for gen, b, n, m in (("U", 8, 4096, 1024), ("D", 8, 4096, 1024), ("D", 4, 8192, 1024), ("S", 8, 2048, 700),
                         ("D", 8, 1024, 1024), ("D", 2, 8192, 512)):
        fps(f"fps_chains/{gen}_{b}_{n}_{m}", t(W.DISTRIBUTIONS[gen](b, n, 35)), m, 128)
    for gen, b, n, m in (("U", 8, 4096, 1024), ("D", 4, 8192, 1024), ("S", 32, 1024, 512), ("U", 2, 16384, 2048), ("D", 1, 65536, 1024)):
        fps(f"fps/{gen}_{b}_{n}_{m}", t(W.DISTRIBUTIONS[gen](b, n, 33)), m, 128)
    for gen, b, n, m in (("U", 1, 262144, 640), ("D", 2, 262144, 512), ("U", 2, 131073, 512), ("U", 8, 65536, 1024), ("D", 8, 16384, 2048)):
        fps(f"fps_large/{gen}_{b}_{n}_{m}", t(W.DISTRIBUTIONS[gen](b, n, 118)), m, 128)

    for gen, b, n, m, r, s in (("U", 8, 4096, 1024, 0.1, 32), ("D", 4, 8192, 1024, 0.1, 32), ("S", 8, 1024, 512, 0.4, 128),
                               ("S", 8, 512, 128, 0.8, 128)):
        xyz = t(W.DISTRIBUTIONS[gen](b, n, 45))
        new_xyz = O.refcuda_gather_point(xyz, O.refcuda_fps(m, xyz))
        ridx, rcnt = O.refcuda_query_ball_point(r, s, xyz, new_xyz)
        rows.add(f"bq/{gen}_{b}_{n}_{m}_{r}_{s}", 16, new_xyz=n_(new_xyz), idx=n_(ridx), cnt=n_(rcnt),
                 grouped=n_(O.refcuda_group_point(xyz, ridx)))
    for b, n in ((2, 65536), (1, 262144)):
        x = t(W.cloud_uniform(b, n, 100 + int(np.log2(n))))
        _, nx = farthest_point_sample_and_gather(n // 4, x)
        ridx, rcnt = O.refcuda_query_ball_point(0.1, 32, x, nx)
        rows.add(f"cfg5_bq/{b}_{n}", 64, idx=n_(ridx), cnt=n_(rcnt))
    x = t(W.cloud_uniform(1, 65536, 116))
    ridx, rcnt = O.refcuda_query_ball_point(0.01, 32, x, x[:, ::4].contiguous())
    rows.add("cfg5_bq_sparse", 64, idx=n_(ridx), cnt=n_(rcnt))

    for b, n, m in ((8, 4096, 2048), (2, 100000, 4096), (33, 777, 100)):
        rng = np.random.RandomState(b + n)
        p = t(rng.random_sample((b, n)).astype(np.float32))
        r = t(rng.random_sample((b, m)).astype(np.float32))
        rows.add(f"prob/{b}_{n}_{m}", 256, out=n_(O.refcuda_prob_sample(p, r)))

    c4 = W.CFG4_SEMSEG
    x = t(W.cloud_duplicates(c4["b"], c4["n"], 100))
    levels, cur = {c4["n"]: x}, x
    for L in c4["sa"]:
        cur = gather_point(cur, farthest_point_sample(L["npoint"], cur))
        levels[L["npoint"]] = cur
    for F in c4["fp"]:
        n, m, c = F["n"], F["m"], F["c"]
        x1, x2 = levels[n], levels[m]
        p2 = W.features(c4["b"], m, c, 105)
        rd, ri = O.refcpu_three_nn(n_(x1), n_(x2))
        dist, _ = three_nn(x1, x2)
        d = torch.clamp(dist, min=1e-10)
        w = (1.0 / d) / (1.0 / d).sum(dim=2, keepdim=True)
        rows.add(f"cfg4_fp/{n}_{m}", 8, dist=rd, idx=ri, out=O.refcpu_three_interpolate(p2, ri, n_(w)))

    def knn_ref(k, x1, x2):
        diff = x1.unsqueeze(1) - x2.unsqueeze(2)
        sq = diff * diff
        outi, out = O.refcuda_selection_sort(k, ((sq[..., 0] + sq[..., 1]) + sq[..., 2]).contiguous())
        return n_(out[:, :, :k]), n_(outi[:, :, :k])

    for gen, b, n, m, k in (("U", 4, 4096, 256, 32), ("D", 3, 3000, 200, 32), ("D", 2, 2048, 128, 128), ("S", 2, 1024, 512, 16),
                            ("U", 2, 40, 10, 40), ("U", 2, 70, 10, 64), ("D", 2, 700, 64, 1), ("U", 1, 8192, 128, 3)):
        x1 = t(W.DISTRIBUTIONS[gen](b, n, 120))
        x2 = gather_point(x1, farthest_point_sample(m, x1)) if gen != "U" else t(W.cloud_uniform(b, m, 121))
        val, idx = knn_ref(k, x1, x2)
        rows.add(f"knn/{gen}_{b}_{n}_{m}_{k}", 16, val=val, idx=idx)
    x1 = t(W.cloud_duplicates(32, 4096, 122))
    x2 = gather_point(x1, farthest_point_sample(1024, x1))
    parts = [knn_ref(32, x1[s:s + 8].contiguous(), x2[s:s + 8].contiguous()) for s in range(0, 32, 8)]
    rows.add("knn_full", 64, val=np.concatenate([p[0] for p in parts]), idx=np.concatenate([p[1] for p in parts]))

    os.makedirs(outdir, exist_ok=True)
    savez_lzma(os.path.join(outdir, "ref_cuda_cases.npz"), rows)
    print("wrote ref_cuda_cases", len(rows), "arrays")


if __name__ == "__main__":
    for flag, fn in (("--ref-cases-cpu", main_ref_cases_cpu), ("--ref-cases-gpu", main_ref_cases_gpu)):
        if flag in sys.argv:
            sys.argv.remove(flag)
            fn(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(HERE), "tests", "golden"))
            sys.exit(0)
    if "--prob-only" in sys.argv:
        sys.argv.remove("--prob-only")
        main_prob(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(HERE), "gpurun_out", "golden"))
        sys.exit(0)
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(HERE), "gpurun_out", "golden"))
