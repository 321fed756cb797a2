import hashlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _has_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden(name: str):
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    if not os.path.exists(path):
        pytest.skip(f"golden fixture {name}.npz not generated yet (oracle/gen_golden.py)")
    return dict(np.load(path))


def assert_golden_rows(got, g, case: str, output: str) -> None:
    """``got`` equals the reference's output ``case/output`` stored by oracle/gen_golden.py
    (ref_{cpu,cuda}_cases.npz) bit for bit: its stored rows first (a readable diff), then the whole
    output through its shape and the sha256 of its bytes."""
    if hasattr(got, "detach"):
        got = got.detach().cpu().numpy()
    got = np.ascontiguousarray(got)
    key = f"{case}/{output}"
    want = g[key]
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    np.testing.assert_array_equal(got.reshape(got.shape[0] * got.shape[1], -1)[g[f"{case}/pos"]], want)
    assert got.shape == tuple(g[key + ".shape"]), (got.shape, tuple(g[key + ".shape"]))
    assert hashlib.sha256(got.tobytes()).hexdigest() == str(g[key + ".sha256"]), f"{key}: differs outside the stored rows"


def golden_names(prefix: str):
    if not os.path.isdir(GOLDEN_DIR):
        return []
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.startswith(prefix) and f.endswith(".npz"))


@pytest.fixture(scope="session")
def dev():
    import torch
    return torch.device("cuda:0")
