"""ctypes loader for libpn2_b200.so — the thin C-ABI layer between the Python ops and the CUDA
kernels (the same mechanism the reference uses for its own native helper, utils/show3d_balls.py:23).

There is NO CPU fallback: if the library cannot be loaded (and cannot be built), importing the
ops raises; calling an op on a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_size_t, c_ulonglong, c_void_p

from . import _build

_P = c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)   — mirrors include/pn2_api.h
    "pn2_fps": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_fps_scratch_bytes": (c_size_t, [c_int, c_int]),
    "pn2_fps_gather": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_prob_sample": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_gather_point": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_gather_point_grad": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_query_ball_point": (c_int, [c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P]),
    "pn2_query_ball_point_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pn2_query_ball_point_ws": (c_int, [c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "pn2_ball_grid_build": (c_int, [c_int, c_int, c_float, c_int, _P, _P, c_size_t, _P]),
    "pn2_query_ball_point_prebuilt": (c_int, [c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "pn2_group_point": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_group_point_grad": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_selection_sort": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_knn_point": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_three_nn": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_three_interpolate": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_three_interpolate_grad": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_three_interpolate_grad_det_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pn2_three_interpolate_grad_det": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "pn2_fp_interpolate_concat": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    "pn2_group_concat": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int, _P, _P, _P]),
    "pn2_three_nn_interpolate": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    # 16-bit features: leading dtype code (PN2_DTYPE_BF16 / PN2_DTYPE_F16), then the float32 twin's arguments
    "pn2_group_point_h": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_group_point_grad_h": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "pn2_group_concat_h": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_int, _P, _P, _P]),
    "pn2_three_interpolate_h": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_three_interpolate_grad_h": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "pn2_three_interpolate_grad_det_h": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "pn2_three_nn_interpolate_h": (c_int, [c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pn2_fp_interpolate_concat_h": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    "pn2_ball_group_fits": (c_int, [c_int]),
    "pn2_ball_group": (c_int, [c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, c_int, _P]),
    "pn2_sa_layer_device_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "pn2_sa_layer_device": (c_int, [c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, _P, c_int, _P, c_size_t, _P]),
    "pn2_sa_layer_msg_device": (c_int, [c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_int, _P, c_size_t, _P]),
    "pn2_set_sa_consumer_ctas": (None, [c_int]),
    "pn2_sa_layer_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "pn2_sa_layer_host": (c_int, [c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "pn2_api_version": (c_int, []),
    "pn2_error_string": (ctypes.c_char_p, [c_int]),
    "pn2_launch_count": (c_ulonglong, []),
    "pn2_ball_threshold": (c_float, [c_float]),
    "pn2_fps_plan": (c_int, [c_int, c_int, _P, _P, _P]),
    "pn2_fps_cluster_capacity": (c_int, [c_int, c_int, c_int]),
    "pn2_set_fps_config": (None, [c_int, c_int, c_int]),
    "pn2_set_bq_group": (None, [c_int]),
    "pn2_set_bq_mode": (None, [c_int]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load() -> ctypes.CDLL:
    """Load (building first if missing/stale and nvcc is present) libpn2_b200.so. Raises on failure."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    world = int(os.environ.get("WORLD_SIZE", "1") or "1")
    local_rank = int(os.environ.get("LOCAL_RANK", "0") or "0")
    if world > 1:
        # one process per GPU: never race on the build tree.  Local rank 0 checks staleness and rebuilds (the
        # library is published with an atomic rename), then writes a stamp naming the source state it was built
        # from; the other local ranks wait for a stamp that matches the sources THEY see, so a library older
        # than the .cu files is never loaded silently.
        want = _build.source_signature()
        stamp = path + ".stamp"
        if local_rank == 0:
            if _build.is_stale():
                try:
                    _build.build()
                except Exception as e:
                    if not os.path.exists(path):
                        raise ImportError(f"libpn2_b200.so is missing and could not be built: {e}") from e
                    want = "prebuilt"  # no nvcc on this box: the library that travelled is what there is
            tmp = stamp + f".tmp{os.getpid()}"
            with open(tmp, "w") as f:
                f.write(want)
            os.replace(tmp, stamp)
        else:
            import time
            deadline = time.time() + 600
            while time.time() < deadline:
                try:
                    got = open(stamp).read()
                except OSError:
                    got = None
                if got in (want, "prebuilt") and os.path.exists(path):
                    break
                time.sleep(0.2)
            else:
                raise ImportError("libpn2_b200.so was not (re)built by local rank 0 within 10 minutes")
    elif _build.is_stale():
        try:
            _build.build()
        except Exception as e:  # stale-but-present library on a box without nvcc is still usable
            if not os.path.exists(path):
                raise ImportError(f"libpn2_b200.so is missing and could not be built: {e}") from e
    try:
        lib = ctypes.CDLL(path)
    except OSError as e:
        raise ImportError(f"cannot load {path}: {e} — the CUDA extension is required, there is no fallback") from e
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class Pn2Error(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().pn2_error_string(rc)
        raise Pn2Error(f"{what} failed: CUDA error {rc} ({msg.decode() if msg else '?'})")


def launch_count() -> int:
    return int(load().pn2_launch_count())
