"""Time the feature kernels with float32, bfloat16 and float16 features, and one PointNet2SemSeg training step in
float32 against bfloat16 autocast.  Writes profiles/half_features.json (or --out).

Kernel rows: K back-to-back launches of one entry point, captured in a CUDA graph (no host overhead between them),
over input sets rotated so that the inputs of one window total more than the 126 MB L2 -- a single launch between two
events after a flush carries a fixed cost of several microseconds (DESIGN section 4) that would hide the halving.
Reported: microseconds per call (median of 5 windows) and the algorithmic bytes of one call over that time.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from pointnet2_b200 import _lib, nets, workloads as W  # noqa: E402
from pointnet2_b200._tensor import FEATURE_DTYPES  # noqa: E402

DTYPES = {"float32": torch.float32, "bfloat16": torch.bfloat16, "float16": torch.float16}
# (b, n, c, m, s) of tools/concat_bench.py: cfg4 SA1/SA2, cfg3 layer 2 (C = 320) at nsample 32 and 128, cfg4 SA4, MSG
GROUP_SHAPES = [(16, 1024, 64, 256, 32), (16, 256, 128, 64, 32), (32, 512, 320, 128, 32), (32, 512, 320, 128, 128),
                (16, 64, 256, 16, 32), (8, 2048, 67, 512, 32)]
# (b, n, m, c2, c1): the feature-propagation layers of PointNet2SemSeg at cfg4 (16 x 8192) and cfg3 (32 x 512 <- 128)
INTERP_SHAPES = [(16, 8192, 1024, 128, 0), (16, 1024, 256, 256, 128), (16, 256, 64, 256, 256), (32, 512, 128, 320, 64)]
L2_BYTES = 126 << 20


def ptr(t):
    return t.data_ptr() if t is not None else None


class Row:
    def __init__(self, op, shape, dtype):
        self.op, self.shape, self.dtype = op, shape, dtype


def time_graph(calls, k_target=400, windows=5):
    """calls: list of zero-argument launchers (one per rotated input set).  Median microseconds per launch."""
    reps = max(1, math.ceil(k_target / len(calls)))
    for fn in calls:  # warm-up outside the capture (module load, one-time attributes)
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            for fn in calls:
                fn()
    g.replay()
    torch.cuda.synchronize()
    k = reps * len(calls)
    ts = []
    for _ in range(windows):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        e.record()
        e.synchronize()
        ts.append(a.elapsed_time(e) * 1e3 / k)
    ts.sort()
    return ts[len(ts) // 2], k


def nsets_for(input_bytes):
    return max(2, min(64, math.ceil(1.05 * L2_BYTES / max(1, input_bytes))))


def stream():
    return torch.cuda.current_stream().cuda_stream


def kernel_rows(dev):
    lib = _lib.load()
    rows = []

    def run(op, shape, dname, build, bytes_moved):
        dt = DTYPES[dname]
        code = FEATURE_DTYPES[dt]
        try:
            calls, input_bytes = build(dt, code)
            us, k = time_graph(calls)
            rows.append(dict(op=op, shape=shape, dtype=dname, us=round(us, 3), launches=k, input_sets=len(calls),
                             inputs_MB_per_window=round(input_bytes * len(calls) / 2**20, 1),
                             GBps=round(bytes_moved(dt.itemsize) / us / 1e3, 1)))
        except Exception as ex:  # keep the other rows; the failure is part of the result
            rows.append(dict(op=op, shape=shape, dtype=dname, error=f"{type(ex).__name__}: {ex}"))
        print(rows[-1], flush=True)
        torch.cuda.empty_cache()

    g = torch.Generator(device=dev).manual_seed(1)
    for (b, n, c, m, s) in GROUP_SHAPES:
        R = b * m * s
        src = b * min(n, m * s)
        shape = dict(b=b, n=n, c=c, m=m, nsample=s)

        def inputs(dt, with_xyz=False):
            per = b * n * c * dt.itemsize + 4 * R + (12 * b * n if with_xyz else 0)
            sets = []
            for _ in range(nsets_for(per)):
                sets.append((torch.randn((b, n, c), device=dev, generator=g).to(dt),
                             torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32),
                             torch.rand((b, n, 3), device=dev, generator=g) if with_xyz else None))
            return sets, per

        def b_group(dt, code):
            sets, per = inputs(dt)
            out = torch.empty((b, m, s, c), dtype=dt, device=dev)
            if code:
                return [lambda p=p, i=i: lib.pn2_group_point_h(code, b, n, c, m, s, ptr(p), ptr(i), ptr(out), stream())
                        for p, i, _ in sets], per
            return [lambda p=p, i=i: lib.pn2_group_point(b, n, c, m, s, ptr(p), ptr(i), ptr(out), stream())
                    for p, i, _ in sets], per
        for dname in DTYPES:
            run("group_point", shape, dname, b_group, lambda es: 4 * R + src * c * es + R * c * es)

        for xyz_first in (1, 0):
            def b_concat(dt, code, xyz_first=xyz_first):
                sets, per = inputs(dt, with_xyz=True)
                out = torch.empty((b, m, s, 3 + c), dtype=dt, device=dev)
                gx = torch.empty((b, m, s, 3), dtype=torch.float32, device=dev)
                new_xyz = torch.rand((b, m, 3), device=dev, generator=g)
                fn = (lambda *a: lib.pn2_group_concat_h(code, *a)) if code else lib.pn2_group_concat
                return [lambda p=p, i=i, x=x: fn(b, n, c, m, s, ptr(x), ptr(new_xyz), ptr(p), ptr(i), xyz_first, ptr(out),
                                                 ptr(gx), stream()) for p, i, x in sets], per
            for dname in DTYPES:
                run("group_concat_xyz_first" if xyz_first else "group_concat_feat_first", shape, dname, b_concat,
                    lambda es: 4 * R + src * (c * es + 12) + R * (c + 3) * es + 12 * R)

        def b_ggrad(dt, code):
            per = R * c * dt.itemsize + 4 * R
            sets = [(torch.randn((b, m, s, c), device=dev, generator=g).to(dt),
                     torch.randint(0, n, (b, m, s), device=dev, generator=g, dtype=torch.int32)) for _ in range(nsets_for(per))]
            gp = torch.zeros((b, n, c), dtype=torch.float32, device=dev)  # accumulates across launches: timing only
            if code:
                return [lambda go=go, i=i: lib.pn2_group_point_grad_h(code, b, n, c, m, s, ptr(go), ptr(i), ptr(gp), stream())
                        for go, i in sets], per
            return [lambda go=go, i=i: lib.pn2_group_point_grad(b, n, c, m, s, ptr(go), ptr(i), ptr(gp), stream())
                    for go, i in sets], per
        for dname in DTYPES:
            run("group_point_grad", shape, dname, b_ggrad, lambda es: R * c * es + 4 * R + 4 * b * n * c)

    for (b, n, m, c2, c1) in INTERP_SHAPES:
        shape = dict(b=b, n=n, m=m, c2=c2, c1=c1)

        def nn_inputs():
            xyz1 = torch.rand((b, n, 3), device=dev, generator=g)
            xyz2 = torch.rand((b, m, 3), device=dev, generator=g)
            dist, idx = torch.empty((b, n, 3), device=dev), torch.empty((b, n, 3), dtype=torch.int32, device=dev)
            _lib.check(lib.pn2_three_nn(b, n, m, ptr(xyz1), ptr(xyz2), ptr(dist), ptr(idx), stream()), "three_nn")
            r = 1.0 / dist.clamp(min=1e-10)
            return xyz1, xyz2, idx, (r / r.sum(2, keepdim=True)).contiguous()

        xyz1, xyz2, idx, w = nn_inputs()

        def b_interp(dt, code):
            per = b * m * c2 * dt.itemsize + 24 * b * n
            sets = [torch.randn((b, m, c2), device=dev, generator=g).to(dt) for _ in range(nsets_for(per))]
            out = torch.empty((b, n, c2), dtype=dt, device=dev)
            fn = (lambda *a: lib.pn2_three_interpolate_h(code, *a)) if code else lib.pn2_three_interpolate
            return [lambda p=p: fn(b, m, c2, n, ptr(p), ptr(idx), ptr(w), ptr(out), stream()) for p in sets], per
        for dname in DTYPES:
            run("three_interpolate", shape, dname, b_interp, lambda es: b * m * c2 * es + 24 * b * n + b * n * c2 * es)

        def b_fp(dt, code):
            per = b * m * c2 * dt.itemsize + b * n * c1 * dt.itemsize + 12 * b * (n + m)
            sets = [(torch.randn((b, m, c2), device=dev, generator=g).to(dt),
                     torch.randn((b, n, c1), device=dev, generator=g).to(dt) if c1 else None) for _ in range(nsets_for(per))]
            out = torch.empty((b, n, c2 + c1), dtype=dt, device=dev)
            fn = (lambda *a: lib.pn2_fp_interpolate_concat_h(code, *a)) if code else lib.pn2_fp_interpolate_concat
            return [lambda p2=p2, p1=p1: fn(b, n, m, c2, c1, ptr(xyz1), ptr(xyz2), ptr(p1), ptr(p2), ptr(out), stream())
                    for p2, p1 in sets], per
        for dname in DTYPES:
            run("fp_interpolate_concat", shape, dname, b_fp,
                lambda es: 12 * b * (n + m) + b * m * c2 * es + b * n * c1 * es + b * n * (c2 + c1) * es)

        def grad_sets(dt):
            per = b * n * c2 * dt.itemsize + 24 * b * n
            return [torch.randn((b, n, c2), device=dev, generator=g).to(dt) for _ in range(nsets_for(per))], per

        def b_igrad(dt, code):
            sets, per = grad_sets(dt)
            gp = torch.zeros((b, m, c2), dtype=torch.float32, device=dev)
            fn = (lambda *a: lib.pn2_three_interpolate_grad_h(code, *a)) if code else lib.pn2_three_interpolate_grad
            return [lambda go=go: fn(b, n, c2, m, ptr(go), ptr(idx), ptr(w), ptr(gp), stream()) for go in sets], per
        for dname in DTYPES:
            run("three_interpolate_grad", shape, dname, b_igrad, lambda es: b * n * c2 * es + 24 * b * n + 4 * b * m * c2)

        def b_dgrad(dt, code):
            sets, per = grad_sets(dt)
            gp = torch.empty((b, m, c2), dtype=torch.float32, device=dev)
            wsb = int(lib.pn2_three_interpolate_grad_det_workspace_bytes(b, n, m))
            ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
            fn = (lambda *a: lib.pn2_three_interpolate_grad_det_h(code, *a)) if code else lib.pn2_three_interpolate_grad_det
            return [lambda go=go: fn(b, n, c2, m, ptr(go), ptr(idx), ptr(w), ptr(gp), ptr(ws), wsb, stream())
                    for go in sets], per
        for dname in DTYPES:
            run("three_interpolate_grad_det", shape, dname, b_dgrad, lambda es: b * n * c2 * es + 24 * b * n + 4 * b * m * c2)
    return rows


def semseg_step(dev, autocast_dtype, b=16, n=8192, steps=5, passes=5):
    torch.manual_seed(0)
    net = nets.PointNet2SemSeg().to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    xyz = torch.from_numpy(W.cloud_uniform(b, n, 5)).to(dev)
    lab = torch.randint(0, 21, (b, n), device=dev, generator=torch.Generator(device=dev).manual_seed(5))

    def step():
        with torch.autocast("cuda", dtype=autocast_dtype or torch.float32, enabled=autocast_dtype is not None):
            pred, _ = net(xyz)
            loss = torch.nn.functional.cross_entropy(pred.float().reshape(-1, pred.shape[-1]), lab.reshape(-1))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(passes):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            loss = step()
        e.record()
        e.synchronize()
        ts.append(a.elapsed_time(e) / steps)
    ts.sort()
    return dict(ms_per_step=round(ts[len(ts) // 2], 3), passes_ms=[round(t, 3) for t in ts], steps_per_pass=steps,
                final_loss=float(loss.detach()))


def gpu_info():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as ex:
        info["nvidia_smi"] = f"unavailable: {ex}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "half_features.json"))
    ap.add_argument("--skip-net", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("half_features_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    t0 = time.time()
    res = dict(gpu=gpu_info(), method=__doc__.strip(), kernels=kernel_rows(dev))
    if not args.skip_net:
        res["semseg_step_cfg4"] = dict(b=16, n=8192, float32=semseg_step(dev, None),
                                       bfloat16_autocast=semseg_step(dev, torch.bfloat16))
        print(res["semseg_step_cfg4"], flush=True)
    res["gpu_after"] = gpu_info()
    res["wall_s"] = round(time.time() - t0, 1)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
