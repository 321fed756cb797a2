#!/usr/bin/env python
"""bench.py — set-abstraction throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this implementation
    python bench.py --impl reference [...]                         # the reference's CPU path
    torchrun --nproc-per-node N bench.py --gpus N ...              # one rank per GPU (weak scaling)

A "step" is one pass of the hot path — farthest_point_sample + gather_point + query_ball_point +
group_point(xyz) — over one batch of the SSG set-abstraction configuration
(BASELINE.json configs[1]: B=32 N=4096 npoint=1024 nsample=32 radius=0.1, uniform synthetic
clouds).  Prints ONE JSON line (rank 0).

  value      whole-job points/s (B*N per rank per step, summed over ranks / max-over-ranks time),
             inputs resident in HBM, CUDA-event timed per step, L2 flushed between steps.
             One batch at a time; a step is ONE pn2_sa_layer_device call (the ball query + grouping
             run as a programmatically dependent grid while the sampling chain is still going).
  e2e        the same metric through the host-buffer C-ABI call (pn2_sa_layer_host): pinned host
             xyz -> H2D -> layer -> D2H of new_xyz/idx/pts_cnt/grouped_xyz, every step, all inside the
             timed region.  Headline: a stream of batches through SetAbstractionPipeline (--e2e-depth
             in flight, default 3); e2e.serial is one batch in flight; e2e.idx_only is the same pipeline
             for a caller that does not ask for grouped_xyz.
  device_batches_in_flight   secondary: `value`'s graph with --in-flight batches on separate
             streams (one layer occupies 2*b of the 148 SMs).
  roofline   dominant kernel (FPS): algorithmic bytes / its CUDA-event time vs the measured HBM peak.
  kernels_ms the three sequential launches of the same step (per-kernel times; their outputs must
             equal the overlapped layer's bit for bit).
  configs    per-kernel rows for BASELINE.json's other configs (cfg3 MSG stack, cfg4 sem-seg SA+FP,
             cfg5 sweep) at this rank's shard, max over ranks — outside every timed region above.
  reference_cuda   the reference's OWN CUDA kernels (oracle/_ref, unmodified) timed on this box.
  cpu_baseline  the same workload on the host cores (FPS: oracle port — the reference has no CPU
             FPS; ball query + group: the reference's own CPU functions when oracle/_ref travelled).

--dump-outputs DIR writes what the timed device-resident leg returned in its last step (rank 0):
DIR/{fps_idx,new_xyz,idx,pts_cnt,grouped_xyz}.npy, float64 for the index tensors (exact) and float32
for the coordinates, 22 MB at the default workload.  The inputs are seeded, so two builds run with
the same arguments can be compared output for output.

Extra: --report FILE writes per-kernel tables for all BASELINE.json configs; --fps-sweep /
--bq-sweep time kernel variants.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "set-abstraction points/sec"
UNIT = "points/s"
L2_FLUSH_BYTES = 256 << 20  # > 126 MB L2
REPEATS = 3  # passes of K steps for the legs timed with ONE event pair around host-driven submission (median reported)


# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()  # the exact process we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
def cpu_cores() -> int:
    """Host CPUs this process can really use: the affinity mask, capped by the cgroup CPU quota (a
    container that shows 128 CPUs with a 16-CPU quota is throttled when 128 workers run)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:  # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    if quota is None:
        try:  # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(quota + 0.999)))
    return n


# The CPU legs keep EVERY host core busy: the reference's functions are single-threaded per call, so
# the unit of parallel work is one cloud (FPS is a serial chain per cloud), and clouds of several
# batches are in flight at once — worker processes (no GIL), forked before the timed region.
_CPU = {}


def _cpu_one_cloud(i: int) -> int:
    """One cloud through the hot path on the host: FPS (C restatement — the reference registers FPS
    for the GPU only, tf_sampling.cpp:123) + gather + ball query + group (the reference's own CPU
    functions from oracle/_ref when they were built, test/query_ball_point.cpp:19-66)."""
    O, xyz, c = _CPU["O"], _CPU["xyz"], _CPU["cfg"]
    cl = xyz[i % xyz.shape[0]][None]
    idx = O.oracle_fps(c["npoint"], cl)
    new_xyz = O.oracle_gather_point(cl, idx)
    if _CPU["use_ref"]:
        bi = O.refcpu_query_ball_point(c["radius"], c["nsample"], cl, new_xyz)
        g = O.refcpu_group_point(cl, bi)
    else:
        bi, _ = O.oracle_query_ball_point(c["radius"], c["nsample"], cl, new_xyz, use_fma=False)
        g = O.oracle_group_point(cl, bi)
    return int(g.shape[1])


def _cpu_setup(cfg):
    from oracle import oracle as O
    from pointnet2_b200 import workloads as W
    use_ref = O.have_refcpu()
    O.lib()
    if use_ref:
        O.refcpu()
    _CPU.update(O=O, cfg=cfg, use_ref=use_ref, xyz=W.DISTRIBUTIONS[cfg["dist"]](cfg["b"], cfg["n"], cfg["seed"]))
    return use_ref


def cpu_throughput(cfg, steps: int, warmup: int):
    """points/s of `steps` batches of the workload on the host at the worker count that serves it
    best; returns (value, seconds, workers, use_ref, single_core_value, calibration)."""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor
    use_ref = _cpu_setup(cfg)
    cpus = cpu_cores()
    b = cfg["b"]
    t1 = time.perf_counter()  # the faithful single-threaded figure first (also warms the libraries)
    for i in range(2):
        _cpu_one_cloud(i)
    one_core = 2 * cfg["n"] / (time.perf_counter() - t1)
    ctx = mp.get_context("fork")

    def rate(ex, workers, tasks):
        chunk = max(1, tasks // (8 * workers))
        t0 = time.perf_counter()
        list(ex.map(_cpu_one_cloud, range(tasks), chunksize=chunk))
        el = time.perf_counter() - t0
        return tasks * cfg["n"] / el, el

    # "all the host threads it can use": a container may show more CPUs than it is allowed to run
    # (quota, busy neighbours), so the worker count is calibrated — the best of a few candidates wins
    cands = sorted({max(1, cpus), max(1, cpus // 2), max(1, cpus // 4), max(1, min(cpus, b)), max(1, min(cpus, 16))}, reverse=True)
    calib = {}
    for w in cands:
        with ProcessPoolExecutor(max_workers=w, mp_context=ctx) as ex:
            rate(ex, w, w)                      # spawn + warm every worker
            calib[w], _ = rate(ex, w, 3 * w)
    workers = max(calib, key=calib.get)
    with ProcessPoolExecutor(max_workers=workers, mp_context=ctx) as ex:
        rate(ex, workers, max(workers, max(warmup, 1) * b))
        value, el = rate(ex, workers, steps * b)
    return value, el, workers, use_ref, one_core, {"host_cpus": cpus, "points_per_s_by_workers": {str(k): round(v) for k, v in calib.items()}}


def _cpu_sample_text(cfg, steps, el, cores, use_ref):
    return (f"{steps} batches of {cfg['name']} ({cfg['b']}x{cfg['n']} pts each) in {el:.2f}s on {cores} worker processes "
            f"(the best of the calibrated worker counts; one cloud per task, {steps * cfg['b']} tasks, batches overlap); FPS = C restatement of "
            f"tf_sampling_g.cu:105-170 (the reference has no CPU FPS); ball query+group = "
            + ("the reference's CPU functions test/query_ball_point.cpp:19-66 (oracle/_ref)" if use_ref else "oracle C restatement"))


def cpu_baseline(cfg, budget_s: float = 12.0):
    """The CPU arm as a child process (this process holds a CUDA context: no fork from here)."""
    steps = 40
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", "3"],
                       capture_output=True, text=True, timeout=max(120.0, 20 * budget_s),
                       env={k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")})
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"error": (r.stderr or "no output")[-300:]}
    return json.loads(lines[-1])["cpu_baseline"]


# ------------------------------------------------------------------------------------------------
def run_reference_arm(args, cfg):
    """--impl reference: the reference's CPU implementation of the path on ALL host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # other ranks exit 0 without work
    value, el, cores, use_ref, one_core, calib = cpu_throughput(cfg, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, 1),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "single_core_value": one_core, "calibration": calib,
                             "kind": "port",  # FPS dominates the CPU time and the reference has no CPU FPS (GPU-only op)
                             "sample": _cpu_sample_text(cfg, args.steps, el, cores, use_ref)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(cfg, world):
    """Identical in both arms (the driver compares it key by key)."""
    return {"workload": f"{cfg['name']}: SSG SA layer FPS+gather_point+query_ball_point+group_point(xyz), "
                        f"B={cfg['b']}/GPU N={cfg['n']} npoint={cfg['npoint']} nsample={cfg['nsample']} radius={cfg['radius']}",
            "global_batch": cfg["b"] * world, "points_per_cloud": cfg["n"], "parallelism": f"dp{world} (clouds sharded, no collective)",
            "distribution": "uniform [0,1)^3, seed 100+rank", "l2": f"flushed between steps ({L2_FLUSH_BYTES >> 20} MiB memset, untimed)"}


# ------------------------------------------------------------------------------------------------
def run_reference_cuda_arm(args, cfg):
    """--impl reference_cuda (child of the product arm, rank 0 only): the reference's OWN CUDA kernels
    (tf_sampling_g.cu:105-181,203-208; tf_grouping_g.cu:3-57,125-136), rebuilt unmodified for sm_100a
    into oracle/_ref, timed with CUDA events on this box at the driver line's workload.  A reported
    comparator like cpu_baseline — never part of the product's timed region."""
    import torch
    from ctypes import c_float, c_int, c_void_p

    from oracle import oracle as O
    from pointnet2_b200 import workloads as W
    if not O.have_refcuda():
        print(json.dumps({"reference_cuda": {"unavailable": "oracle/_ref CUDA libraries are not in this tree"}}), flush=True)
        return
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    samp, grp = O.refcuda()
    b, n, m, s, r = cfg["b"], cfg["n"], cfg["npoint"], cfg["nsample"], cfg["radius"]
    xyz = torch.from_numpy(W.DISTRIBUTIONS[cfg["dist"]](b, n, cfg["seed"])).to(dev)
    temp = torch.empty((32, n), dtype=torch.float32, device=dev)
    fi = torch.zeros((b, m), dtype=torch.int32, device=dev)
    nx = torch.empty((b, m, 3), dtype=torch.float32, device=dev)
    idx = torch.zeros((b, m, s), dtype=torch.int32, device=dev)
    cnt = torch.zeros((b, m), dtype=torch.int32, device=dev)
    g = torch.empty((b, m, s, 3), dtype=torch.float32, device=dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    P = lambda t: c_void_p(t.data_ptr())  # noqa: E731
    ops = [
        ("farthestpointsamplingLauncher", lambda: samp._Z29farthestpointsamplingLauncheriiiPKfPfPi(c_int(b), c_int(n), c_int(m), P(xyz), P(temp), P(fi))),
        ("gatherpointLauncher", lambda: samp._Z19gatherpointLauncheriiiPKfPKiPf(c_int(b), c_int(n), c_int(m), P(xyz), P(fi), P(nx))),
        ("queryBallPointLauncher", lambda: grp._Z22queryBallPointLauncheriiifiPKfS0_PiS1_(c_int(b), c_int(n), c_int(m), c_float(r), c_int(s), P(xyz), P(nx), P(idx), P(cnt))),
        ("groupPointLauncher", lambda: grp._Z18groupPointLauncheriiiiiPKfPKiPf(c_int(b), c_int(n), c_int(3), c_int(m), c_int(s), P(xyz), P(idx), P(g))),
    ]
    # the reference launches on the legacy default stream: time there
    st = torch.cuda.default_stream(dev)
    steps = max(3, min(args.steps, 10))
    ms = {k: [] for k, _ in ops}
    with torch.cuda.stream(st):
        for it in range(3 + steps):
            flush.zero_()
            for name, fn in ops:
                a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                fn()
                z.record(st)
                z.synchronize()
                if it >= 3:
                    ms[name].append(a.elapsed_time(z))
    per = {k: statistics.median(v) for k, v in ms.items()}
    total = sum(per.values())
    print(json.dumps({"reference_cuda": {
        "what": "the reference's own CUDA kernels (tf_sampling_g.cu, tf_grouping_g.cu), nvcc -O2 for sm_100a, unmodified, "
                "legacy default stream, CUDA events, L2 flushed before each step",
        "kernels_ms": per, "ms_per_step": total, "value": b * n / (total * 1e-3), "unit": UNIT, "steps": steps,
        "workload": workload_config(cfg, 1)["workload"]}}), flush=True)


def child_json(argv, key, timeout=600.0):
    """Run bench.py in a child process (fresh CUDA context / no fork from a CUDA process) and pick `key` from its JSON line."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__)] + argv, capture_output=True, text=True, timeout=timeout,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")})
    except subprocess.TimeoutExpired:
        return {"error": f"timed out after {timeout:.0f}s"}
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"error": (r.stderr or "no output")[-300:]}
    return json.loads(lines[-1]).get(key, {"error": f"no {key} in the child's line"})


# ------------------------------------------------------------------------------------------------
def dump_outputs(out_dir: str, o: dict) -> None:
    """The layer's outputs as a caller receives them: index tensors as float64 (exact), coordinates as float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, key in (("fps_idx", "fps_idx"), ("new_xyz", "new_xyz"), ("idx", "idx"), ("pts_cnt", "cnt"), ("grouped_xyz", "grouped")):
        a = o[key].cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype.kind == "i" else np.float32))


def run_b200_arm(args, cfg):
    import ctypes

    import torch
    import torch.distributed as dist

    from pointnet2_b200 import _lib, numa, workloads as W
    from pointnet2_b200.host import SetAbstractionHost, SetAbstractionPipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa.bind_cpus(dev)  # one process per GPU: run (and first-touch pinned memory) on the GPU's own socket
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    lib = _lib.load()
    b, n, m, s, r = cfg["b"], cfg["n"], cfg["npoint"], cfg["nsample"], cfg["radius"]
    xyz_np = W.DISTRIBUTIONS[cfg["dist"]](b, n, cfg["seed"] + rank)
    xyz = torch.from_numpy(xyz_np).to(dev)

    def out_buffers():
        return dict(fps_idx=torch.empty((b, m), dtype=torch.int32, device=dev), new_xyz=torch.empty((b, m, 3), dtype=torch.float32, device=dev),
                    idx=torch.empty((b, m, s), dtype=torch.int32, device=dev), cnt=torch.empty((b, m), dtype=torch.int32, device=dev),
                    grouped=torch.empty((b, m, s, 3), dtype=torch.float32, device=dev))

    seq, fus = out_buffers(), out_buffers()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    bq_ws_bytes = int(lib.pn2_query_ball_point_workspace_bytes(b, n))  # caller-provided scratch for the grid path
    bq_ws = torch.empty(bq_ws_bytes, dtype=torch.uint8, device=dev) if bq_ws_bytes else None
    dws_bytes = int(lib.pn2_sa_layer_device_workspace_bytes(b, n, m, s))
    st = torch.cuda.current_stream(dev)
    sp = st.cuda_stream

    def step_sequential(ev=None):
        """The four reference ops as three separate launches (the per-kernel breakdown and the
        bit-identity check of the overlapped layer)."""
        o = seq
        if ev:
            ev[0].record(st)
        rc = lib.pn2_fps_gather(b, n, m, xyz.data_ptr(), None, o["fps_idx"].data_ptr(), o["new_xyz"].data_ptr(), sp)
        if ev:
            ev[1].record(st)
        rc |= lib.pn2_query_ball_point_ws(b, n, m, r, s, xyz.data_ptr(), o["new_xyz"].data_ptr(), o["idx"].data_ptr(), o["cnt"].data_ptr(),
                                          bq_ws.data_ptr() if bq_ws is not None else None, bq_ws_bytes, sp)
        if ev:
            ev[2].record(st)
        rc |= lib.pn2_group_point(b, n, 3, m, s, xyz.data_ptr(), o["idx"].data_ptr(), o["grouped"].data_ptr(), sp)
        if ev:
            ev[3].record(st)
        if rc:
            raise RuntimeError(f"kernel launch failed rc={rc}")

    def layer(o, ws, stream_ptr):
        """The product's layer call: FPS+gather with the ball query + grouping overlapped on the idle SMs."""
        rc = lib.pn2_sa_layer_device(b, n, m, r, s, xyz.data_ptr(), o["fps_idx"].data_ptr(), o["new_xyz"].data_ptr(), o["idx"].data_ptr(),
                                     o["cnt"].data_ptr(), o["grouped"].data_ptr(), 0, ws.data_ptr() if ws is not None else None,
                                     dws_bytes, stream_ptr)
        if rc:
            raise RuntimeError(f"pn2_sa_layer_device failed rc={rc}")

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- per-kernel breakdown (sequential launches on one stream, events between the ops) -----
    for _ in range(args.warmup):
        flush.zero_()
        step_sequential()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    barrier()
    for k in range(args.steps):
        flush.zero_()
        step_sequential(evs[k])
    barrier()
    t_fps = [e[0].elapsed_time(e[1]) for e in evs]
    t_bq = [e[1].elapsed_time(e[2]) for e in evs]
    t_grp = [e[2].elapsed_time(e[3]) for e in evs]
    t_seq = [e[0].elapsed_time(e[3]) for e in evs]

    # ---- device-resident leg (the `value`): ONE pn2_sa_layer_device call per step — two launches, the
    #      second a programmatically dependent grid that consumes centroids while the sampling chain
    #      runs — replayed as a CUDA graph when capture works ----
    dws = torch.empty(dws_bytes, dtype=torch.uint8, device=dev) if dws_bytes else None
    layer(fus, dws, sp)  # loads modules / sets function attributes outside any capture
    torch.cuda.synchronize(dev)
    l0 = _lib.launch_count()
    layer(fus, dws, sp)
    torch.cuda.synchronize(dev)
    launches_per_step = _lib.launch_count() - l0
    graph, launch_mode = None, "direct launches"
    try:
        g = torch.cuda.CUDAGraph()
        cap = torch.cuda.Stream(dev)
        with torch.cuda.graph(g, stream=cap):
            layer(fus, dws, torch.cuda.current_stream(dev).cuda_stream)
        g.replay()
        torch.cuda.synchronize(dev)
        graph, launch_mode = g, "one CUDA graph per step"
    except Exception as e:  # noqa: BLE001 — fall back to direct launches, say so in the JSON
        launch_mode += f" (graph capture failed: {type(e).__name__})"
        torch.cuda.synchronize(dev)

    def run_step():
        if graph is not None:
            graph.replay()
        else:
            layer(fus, dws, sp)

    for _ in range(args.warmup):
        flush.zero_()
        run_step()
    sev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    for k in range(args.steps):
        flush.zero_()
        sev[k][0].record(st)
        run_step()
        sev[k][1].record(st)
    barrier()
    launches = launches_per_step * args.steps
    t_step = [a.elapsed_time(bb) for a, bb in sev]
    total_ms = max_over_ranks(sum(t_step))
    value = world * b * n * args.steps / (total_ms * 1e-3)
    # the overlapped layer must produce exactly what the three sequential launches produced
    same_dev = all(bool(torch.equal(fus[k], seq[k])) for k in seq)

    # ---- secondary: several independent batches in flight (one layer occupies 2*b of the 148 SMs).
    #      Reported beside `value` (which stays one batch at a time), never instead of it. ----
    inflight = None
    graph_everywhere = max_over_ranks(0.0 if graph is not None else 1.0) == 0.0
    if graph_everywhere and args.in_flight > 1:
        try:
            lanes = []
            for _ in range(args.in_flight):
                bufs = out_buffers()
                lws = torch.empty(dws_bytes, dtype=torch.uint8, device=dev) if dws_bytes else None
                ls = torch.cuda.Stream(dev)
                lg = torch.cuda.CUDAGraph()
                with torch.cuda.graph(lg, stream=ls):
                    layer(bufs, lws, torch.cuda.current_stream(dev).cuda_stream)
                lanes.append((lg, ls, bufs))

            def run_lanes(steps, t0=None):
                for lg, ls, _ in lanes:
                    if t0 is not None:
                        ls.wait_event(t0)
                for k in range(steps):
                    lg, ls, _ = lanes[k % len(lanes)]
                    with torch.cuda.stream(ls):
                        flush.zero_()
                        lg.replay()

            run_lanes(max(args.warmup, len(lanes)))
            passes = []
            for _ in range(REPEATS):  # one event pair around K steps is exposed to host hiccups: median of REPEATS passes
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(dev)  # no collective inside this try: a failing rank must not strand the others
                q0.record(st)
                run_lanes(args.steps, q0)
                for _, ls, _ in lanes:
                    st.wait_stream(ls)
                q1.record(st)
                torch.cuda.synchronize(dev)
                launches += launches_per_step * args.steps
                passes.append(q0.elapsed_time(q1))
            fl_local = statistics.median(passes)
            lanes_same = all(bool(torch.equal(bf["idx"], seq["idx"])) and bool(torch.equal(bf["grouped"], seq["grouped"])) for _, _, bf in lanes)
            inflight = {"batches_in_flight": len(lanes), "unit": UNIT, "outputs_match_sequential": lanes_same,
                        "timing": f"one event pair around all {args.steps} steps, L2 flush inside; median of {REPEATS} such passes",
                        "passes_ms_per_step": [round(t / args.steps, 5) for t in passes]}
        except Exception as e:  # noqa: BLE001 — secondary number only
            fl_local = float("inf")
            inflight = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.synchronize(dev)
        fl_ms = max_over_ranks(fl_local)  # every rank takes part whether or not its own leg succeeded
        if fl_ms != float("inf") and "error" not in inflight:
            inflight.update(value=world * b * n * args.steps / (fl_ms * 1e-3), ms_per_step=fl_ms / args.steps)
        elif "error" not in inflight:
            inflight = {"error": "the leg failed on another rank"}

    # ---- end-to-end, one batch in flight: host buffers through the C-ABI host call --------------------------
    sess = SetAbstractionHost(b, n, m, r, s, device=dev)
    sess.h_xyz.numpy()[...] = xyz_np
    for _ in range(args.warmup):
        flush.zero_()
        sess.launch(st)
    e2e_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches1 = _lib.launch_count()
    barrier()
    for k in range(args.steps):
        flush.zero_()
        e2e_ev[k][0].record(st)
        sess.launch(st)
        e2e_ev[k][1].record(st)
    barrier()
    launches += _lib.launch_count() - launches1
    e2e_serial_ms = max_over_ranks(sum(a.elapsed_time(bb) for a, bb in e2e_ev))
    e2e_serial_value = world * b * n * args.steps / (e2e_serial_ms * 1e-3)
    same = bool((sess.h_idx.to(dev) == seq["idx"]).all()) and bool((sess.h_new_xyz.to(dev) == seq["new_xyz"]).all())

    # ---- end-to-end, the headline: the same host-buffer call for a STREAM of batches — a ring of `depth`
    #      sessions on private streams (SetAbstractionPipeline).  Every step copies its input from pinned
    #      host memory and its results back; the L2 flush runs inside the timed region. ----
    def e2e_pipeline(want_grouped):
        nonlocal launches
        pipe = SetAbstractionPipeline(b, n, m, r, s, depth=args.e2e_depth, device=dev, want_grouped=want_grouped)
        for sl in pipe.slots:
            sl.h_xyz.numpy()[...] = xyz_np

        def run_pipe(steps, t0=None):
            if t0 is not None:
                for ps in pipe.streams:
                    ps.wait_event(t0)
            for _ in range(steps):
                if pipe.full():
                    pipe.collect()
                with torch.cuda.stream(pipe.streams[pipe._next]):
                    flush.zero_()
                pipe.submit()
            while pipe.pending():
                pipe.collect()

        run_pipe(max(args.warmup, pipe.depth))
        passes = []
        for _ in range(REPEATS):
            # The region spans K steps of host-driven submission, so one host hiccup (a GC pause, a descheduled thread:
            # 5-60 ms seen on the GPU boxes while every batch's own GPU time stayed at 0.55 ms) lands in it: each pass
            # times EXACTLY K steps, max over ranks, and the median of REPEATS passes is reported (all of them listed).
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l2 = _lib.launch_count()
            barrier()
            p0.record(st)
            run_pipe(args.steps, p0)
            for ev in pipe.done:
                st.wait_event(ev)
            p1.record(st)
            barrier()
            launches += _lib.launch_count() - l2
            passes.append(max_over_ranks(p0.elapsed_time(p1)))
        ms = statistics.median(passes)
        ok = all(bool((sl.h_idx.to(dev) == seq["idx"]).all()) and bool((sl.h_new_xyz.to(dev) == seq["new_xyz"]).all())
                 and (not want_grouped or bool((sl.h_grouped_xyz.to(dev) == seq["grouped"]).all())) for sl in pipe.slots)
        return ms, ok, pipe.h2d_bytes, pipe.d2h_bytes, [round(t / args.steps, 5) for t in passes]

    import gc
    gc.collect()
    gc.disable()  # no collector pauses inside the host-driven timed regions
    e2e_ms, same_pipe, h2d_bytes, d2h_bytes, e2e_passes = e2e_pipeline(True)
    e2e_value = world * b * n * args.steps / (e2e_ms * 1e-3)
    lean_ms, same_lean, _, lean_d2h, lean_passes = e2e_pipeline(False)
    gc.enable()
    clocks = sampler.stop() if rank == 0 else None

    # ---- the other BASELINE configs (cfg3 MSG stack, cfg4 sem-seg SA+FP, cfg5 sweep) at this rank's shard,
    #      per kernel, max over ranks — outside every timed region above ----
    configs_block = None
    if not args.no_configs:
        import bench_report
        peak_c, kind_c = measured_peaks()
        try:
            rows = bench_report.config_rows(torch, lib, dev, flush, peak_c, kind_c, world=world, rank=rank, reps=5, full=False, echo=False)
            ms_vec = torch.tensor([rw["ms"] for rw in rows], dtype=torch.float64, device=dev)
            ok_flag = 0.0
        except Exception as e:  # noqa: BLE001
            rows, ms_vec, ok_flag = [], torch.zeros(1, dtype=torch.float64, device=dev), 1.0
            configs_block = {"error": f"{type(e).__name__}: {e}"}
        if max_over_ranks(ok_flag) == 0.0:
            if world > 1:
                dist.all_reduce(ms_vec, op=dist.ReduceOp.MAX)
            out_rows = []
            for rw, ms_v in zip(rows, ms_vec.tolist()):
                nbytes = rw["algorithmic_MB"] * 1e6
                o = {"config": rw["config"], "kernel": rw["kernel"], "ms": ms_v, "GBps_per_gpu": nbytes / (ms_v * 1e-3) / 1e9,
                     "frac_of_peak": nbytes / (ms_v * 1e-3) / 1e9 / peak_c}
                for k2 in ("us_per_iter", "fp32_issue_frac_of_gpu", "mean_cnt"):
                    if k2 in rw:
                        o[k2] = rw[k2] * (rw["ms"] / ms_v if k2 == "fp32_issue_frac_of_gpu" else (ms_v / rw["ms"] if k2 == "us_per_iter" else 1.0))
                if "points_per_s" in rw:
                    o["points_per_s_all_gpus"] = world * rw["points_per_s"] * rw["ms"] / ms_v
                out_rows.append(o)
            configs_block = {"what": "per kernel: CUDA events, L2 flushed before each timed launch, median of 5 (2-3 for N >= 65536), max over ranks; "
                                     f"cfg3 B=32/GPU, cfg4 B={max(1, 16 // world)}/GPU, cfg5 B={max(1, 8 // world)}/GPU",
                             "peak": f"{peak_c} GB/s of {kind_c}", "rows": out_rows}
        elif configs_block is None:
            configs_block = {"error": "the configs block failed on another rank"}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, fus)  # no later leg writes `fus`: it holds the last timed step's outputs
    if rank == 0:
        pt, pp, pc = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        lib.pn2_fps_plan(b, n, ctypes.byref(pt), ctypes.byref(pp), ctypes.byref(pc))
        kinds = {1: "fps_cta_kernel", 0: "fps_global_kernel"}
        # chain of the sampling kernel: the packed FP32x2 / value-only update is the library's built-in choice wherever
        # it is instantiated (>= 8 points per thread for one CTA per cloud, a multiple of 4 for clusters)
        env_chain = os.environ.get("PN2_FPS_PACKED" if pc.value == 1 else "PN2_FPS_PACKED_CLUSTER", "1")
        packed_chain = env_chain != "0" and (pp.value >= 8 if pc.value == 1 else (pc.value > 1 and pp.value % 4 == 0))
        fps_kernel = (f"{kinds.get(pc.value, 'fps_cluster_kernel')}<{pp.value},{pt.value}{',1' if packed_chain else ''}>"
                      + (f" cluster={pc.value}" if pc.value > 1 else "") + (" packed chain" if packed_chain else ""))
        peak, peak_kind = measured_peaks()
        fps_ms = statistics.mean(t_fps)
        fps_bytes = W.bytes_fps(b, n, m, with_new_xyz=True)
        achieved = fps_bytes / (fps_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("fps_dram_bytes_per_launch")
                traffic_src = "profiles/ncu_traffic.json: " + tj.get("source", "ncu --set full capture of this kernel") + " (not re-measured in this run)"
            except Exception:
                traffic = None
        layer_bytes = W.bytes_sa_layer(b, n, m, s)
        step_ms = statistics.mean(t_step)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(cfg, world),
            "launch": f"pn2_sa_layer_device: sampling kernel + programmatically dependent ball-query/grouping grid ({launches_per_step} launches per step), {launch_mode}",
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms / args.steps, "outputs_match_device_leg": same and same_pipe,
                    "mode": f"stream of batches, {args.e2e_depth} in flight (SetAbstractionPipeline -> pn2_sa_layer_host); one event pair around all "
                            f"{args.steps} steps, L2 flush inside; median of {REPEATS} such passes",
                    "passes_ms_per_step": e2e_passes,
                    "serial": {"value": e2e_serial_value, "ms_per_step": e2e_serial_ms / args.steps,
                               "mode": "one batch in flight (SetAbstractionHost); per-step event pairs, L2 flush between"},
                    "idx_only": {"value": world * b * n * args.steps / (lean_ms * 1e-3), "ms_per_step": lean_ms / args.steps,
                                 "d2h_bytes_per_step": lean_d2h, "outputs_match_device_leg": same_lean, "passes_ms_per_step": lean_passes,
                                 "mode": "same pipeline with grouped_xyz = NULL (new_xyz, idx, pts_cnt come back; the caller regroups xyz[idx] itself)"},
                    "numa": numa.status()},
            "gpu_launches": int(launches),  # this library's kernels inside the timed regions
            "roofline": {"bound": "hbm", "kernel": fps_kernel + " (FPS + fused gather_point)", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_kind": f"of {peak_kind}",
                         "algorithmic_bytes_per_launch": fps_bytes, "ms_per_launch": fps_ms,
                         "note": "FPS is a serial chain of npoint argmax steps: latency/FP32-issue bound, not HBM bound; it is "
                                 f"{100 * fps_ms / step_ms:.0f} % of the step now that the ball query + grouping overlap it",
                         "secondary": {"point_pairs_per_s": b * (m - 1) * n / (fps_ms * 1e-3),
                                       # normalised to the PLAIN chain's 10 scalar instructions per point pair
                                       # (SASS: 3 FADD, FMUL, 2 FFMA, FMNMX, FSETP, FSEL, SEL) so that rounds compare; the
                                       # packed chain issues ~5.5 per pair (3 FP32x2 halves, FMNMX, 0.6 of FMNMX3, search)
                                       "fp32_issue_basis": "10 scalar instructions per point pair (plain chain); the packed chain issues ~5.5",
                                       "fp32_issue_frac_of_gpu": b * (m - 1) * n * 10 / (fps_ms * 1e-3) / (148 * 128 * 1.965e9),
                                       "fp32_issue_frac_of_occupied_sms": b * (m - 1) * n * 10 / (fps_ms * 1e-3) / (min(b, 148) * 128 * 1.965e9),
                                       "whole_layer_GBps": layer_bytes / (step_ms * 1e-3) / 1e9,
                                       "whole_layer_frac": layer_bytes / (step_ms * 1e-3) / 1e9 / peak}},
            "kernels_ms": {"fps_gather": fps_ms, "query_ball_point": statistics.mean(t_bq), "group_point": statistics.mean(t_grp),
                           "step_sequential": statistics.mean(t_seq), "step": step_ms,
                           "overlap_hides_ms": statistics.mean(t_seq) - step_ms,
                           "overlapped_outputs_match_sequential": same_dev,
                           "GBps": {"query_ball_point": W.bytes_ball_query(b, n, m, s) / (statistics.mean(t_bq) * 1e-3) / 1e9,
                                    "group_point": W.bytes_group(b, n, m, s, 3) / (statistics.mean(t_grp) * 1e-3) / 1e9}},
            "device_batches_in_flight": inflight,
            "configs": configs_block,
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["reference_cuda"] = child_json(["--impl", "reference_cuda", "--steps", "10", "--warmup", "3"], "reference_cuda", timeout=300.0)
            line["cpu_baseline"] = cpu_baseline(cfg, budget_s=args.cpu_budget)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference", "reference_cuda"], default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline and reference_cuda children")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg3/cfg4/cfg5 per-kernel block")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--in-flight", type=int, default=4, help="batches in flight in the secondary device-resident leg")
    ap.add_argument("--e2e-depth", type=int, default=3, help="batches in flight in the end-to-end leg")
    ap.add_argument("--report", type=str, default=None, help="write per-kernel tables for all BASELINE configs to this file")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write the timed leg's outputs of its last step to DIR/<name>.npy")
    ap.add_argument("--fps-sweep", action="store_true")
    ap.add_argument("--bq-sweep", action="store_true")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    from pointnet2_b200 import workloads as W
    cfg = dict(W.CFG2_SSG_SA)
    if args.report or args.fps_sweep or args.bq_sweep:
        import bench_report
        bench_report.main(args)
        return
    if args.impl == "reference":
        run_reference_arm(args, cfg)
    elif args.impl == "reference_cuda":
        run_reference_cuda_arm(args, cfg)
    else:
        run_b200_arm(args, cfg)


if __name__ == "__main__":
    main()
