"""CPU checks of the 16-bit feature entry points (pn2_*_h): dtype codes and argument errors are reported without a
launch, and the Python wrappers accept only float32 / bfloat16 / float16 features and float32 coordinates."""
import ctypes

import pytest
import torch

import pointnet2_b200
from pointnet2_b200 import _lib
from pointnet2_b200.pointnet_util import group_and_concat
from pointnet2_b200.tf_interpolate import fp_interpolate_concat, three_nn_interpolate

NULL = ctypes.c_void_p(0)
P = ctypes.c_void_p(256)  # a non-null pointer: never dereferenced, every call below fails its argument checks first


def _calls(dt, b=1, n=8, c=4, m=2, s=2, ptr=P):
    """Every _h entry with otherwise valid sizes."""
    lib = _lib.load()
    return {
        "pn2_group_point_h": lambda: lib.pn2_group_point_h(dt, b, n, c, m, s, ptr, ptr, ptr, NULL),
        "pn2_group_point_grad_h": lambda: lib.pn2_group_point_grad_h(dt, b, n, c, m, s, ptr, ptr, ptr, NULL),
        "pn2_group_concat_h": lambda: lib.pn2_group_concat_h(dt, b, n, c, m, s, ptr, ptr, ptr, ptr, 1, ptr, ptr, NULL),
        "pn2_three_interpolate_h": lambda: lib.pn2_three_interpolate_h(dt, b, m, c, n, ptr, ptr, ptr, ptr, NULL),
        "pn2_three_interpolate_grad_h": lambda: lib.pn2_three_interpolate_grad_h(dt, b, n, c, m, ptr, ptr, ptr, ptr, NULL),
        "pn2_three_interpolate_grad_det_h": lambda: lib.pn2_three_interpolate_grad_det_h(dt, b, n, c, m, ptr, ptr, ptr, ptr,
                                                                                         ptr, 1 << 20, NULL),
        "pn2_three_nn_interpolate_h": lambda: lib.pn2_three_nn_interpolate_h(dt, b, n, m, c, ptr, ptr, ptr, ptr, ptr, ptr,
                                                                             ptr, NULL),
        "pn2_fp_interpolate_concat_h": lambda: lib.pn2_fp_interpolate_concat_h(dt, b, n, m, c, c, ptr, ptr, ptr, ptr, ptr,
                                                                               NULL),
    }


def test_every_half_entry_is_declared_and_covered():
    half = {s for s in _lib.EXPORTED_SYMBOLS if s.endswith("_h")}
    assert half == set(_calls(1))


@pytest.mark.parametrize("dt", [0, 3, 4, -1])
def test_unknown_dtype_codes_are_refused_without_a_launch(dt):
    before = _lib.launch_count()
    for name, call in _calls(dt).items():
        assert call() == 1, name
    for name, call in _calls(dt, b=0).items():  # even an empty call names its dtype
        assert call() == 1, name
    assert _lib.launch_count() == before


@pytest.mark.parametrize("dt", [1, 2])
def test_null_and_negative_arguments_are_refused_without_a_launch(dt):
    before = _lib.launch_count()
    for name, call in _calls(dt, ptr=NULL).items():
        assert call() == 1, name
    for field in ("b", "n", "c", "m"):
        for name, call in _calls(dt, **{field: -1}).items():
            assert call() == 1, (name, field)
    for name, call in _calls(dt, s=-1).items():
        if name.startswith("pn2_group"):
            assert call() == 1, name
    assert _lib.launch_count() == before


def test_feature_dtypes_are_validated():
    x = torch.zeros(1, 8, 3)
    i3 = torch.zeros(1, 4, 3, dtype=torch.int32)
    w = torch.zeros(1, 4, 3)
    with pytest.raises(TypeError, match="float32, torch.bfloat16 or torch.float16"):
        pointnet2_b200.group_point(torch.zeros(1, 8, 4, dtype=torch.float64), i3)
    with pytest.raises(TypeError):
        pointnet2_b200.three_interpolate(torch.zeros(1, 8, 4, dtype=torch.float64), i3, w)
    with pytest.raises(TypeError):
        three_nn_interpolate(x, x, torch.zeros(1, 8, 4, dtype=torch.float64))
    with pytest.raises(TypeError):
        group_and_concat(x, x, torch.zeros(1, 8, 4, dtype=torch.int32), i3)
    with pytest.raises(TypeError):
        fp_interpolate_concat(x, x, None, torch.zeros(1, 8, 4, dtype=torch.float64))


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
def test_coordinates_and_weights_stay_float32(dt):
    # (on a CPU tensor the first coordinate argument is the one that is checked; the others: the GPU tests)
    x, xh = torch.zeros(1, 8, 3), torch.zeros(1, 8, 3, dtype=dt)
    f = torch.zeros(1, 8, 4, dtype=dt)
    i3 = torch.zeros(1, 4, 3, dtype=torch.int32)
    with pytest.raises(TypeError, match="xyz"):
        group_and_concat(xh, x, f, i3)
    with pytest.raises(TypeError, match="xyz1"):
        three_nn_interpolate(xh, x, f)
    with pytest.raises(TypeError):
        pointnet2_b200.three_nn(xh, x)


def test_fp_interpolate_concat_needs_one_feature_dtype():
    x = torch.zeros(1, 8, 3)
    with pytest.raises(TypeError, match="one dtype"):
        fp_interpolate_concat(x, x, torch.zeros(1, 8, 4, dtype=torch.bfloat16), torch.zeros(1, 8, 4))
    with pytest.raises(TypeError, match="one dtype"):
        fp_interpolate_concat(x, x, torch.zeros(1, 8, 4, dtype=torch.float16), torch.zeros(1, 8, 4, dtype=torch.bfloat16))


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
def test_half_features_on_cpu_still_have_no_cpu_path(dt):
    with pytest.raises(RuntimeError, match="no CPU path"):
        pointnet2_b200.group_point(torch.zeros(1, 8, 4, dtype=dt), torch.zeros(1, 4, 3, dtype=torch.int32))
