"""CPU checks of the BVH builds' refusals: the checks RayTracer makes before a device build (mc_ops.validate_device_mesh is
plain torch, so it runs here on CPU tensors), the host build's own checks, and the new entry points' argument errors.  All
of them fire before any allocation or launch, so none needs a GPU."""
import ctypes

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from tensoflow_b200 import build, _lib
    build.build()
    return _lib.load()


def _mesh():
    from tensoflow_b200.synthetic import bumpy_sphere
    return bumpy_sphere(16, 8)


@pytest.mark.parametrize("case,match", [
    ("index-high", "out of range"), ("index-negative", "out of range"), ("nan", "non-finite"), ("inf", "non-finite"),
    ("no-triangles", "empty mesh"), ("no-vertices", "empty mesh"), ("eight", "at least 8"), ("shape", r"\[T, 3\]"),
    ("float-triangles", "int32 / int64"), ("2^31", "2\\^31"), ("beyond-fp32", "non-finite"),
])
def test_device_mesh_checks_raise_before_any_launch(lib, case, match):
    from tensoflow_b200.mc_ops import validate_device_mesh
    v, t = _mesh()
    if case == "index-high":
        t = t.clone()
        t[3, 2] = v.shape[0]
    elif case == "index-negative":
        t = t.long()
        t[0, 0] = -1
    elif case in ("nan", "inf"):
        v = v.clone()
        v[int(t[9, 1]), 1] = float("nan") if case == "nan" else float("inf")
    elif case == "no-triangles":
        t = t[:0]
    elif case == "no-vertices":
        v = v[:0]
    elif case == "eight":
        t = t[:8]
    elif case == "shape":
        t = t.reshape(-1, 6)
    elif case == "float-triangles":
        t = t.float()
    elif case == "beyond-fp32":
        v = v.double()
        v[int(t[4, 0]), 2] = 1e39                                             # finite in float64, inf in the build's fp32
    elif case == "2^31":
        t = torch.zeros(1, 3, dtype=torch.int32).expand(1 << 31, 3)          # a view: no memory behind it
    n0 = lib.tf_launch_count()
    with pytest.raises(RuntimeError, match=match):
        validate_device_mesh(v, t)
    assert lib.tf_launch_count() == n0


def test_too_few_triangles_is_still_an_assertion(lib):
    from tensoflow_b200.mc_ops import validate_device_mesh
    v, t = _mesh()
    with pytest.raises(AssertionError, match="at least 8"):
        validate_device_mesh(v, t[:8])


def test_device_mesh_checks_pass_a_good_mesh(lib):
    from tensoflow_b200.mc_ops import validate_device_mesh
    v, t = _mesh()
    extra = torch.cat([v, torch.full((1, 3), float("nan"))])               # an unreferenced non-finite vertex is allowed
    assert validate_device_mesh(extra, t.long()) == (t.shape[0], v.shape[0] + 1)


@pytest.mark.parametrize("case,match", [("nan", "non-finite"), ("inf", "non-finite"), ("index", "out of range")])
def test_host_build_refuses_before_allocating(lib, case, match):
    """tf_bvh_create checks every referenced vertex and index before it builds or touches the device"""
    from tensoflow_b200.mc_ops import RayTracer
    v, t = (x.numpy().copy() for x in _mesh())
    if case == "index":
        t[5, 0] = v.shape[0]
    else:
        v[t[11, 2], 0] = np.nan if case == "nan" else -np.inf
    n0 = lib.tf_launch_count()
    with pytest.raises(RuntimeError, match=match):
        RayTracer(v, t)
    assert lib.tf_launch_count() == n0


def test_build_entry_points_refuse_bad_arguments(lib):
    n_nodes, ws = ctypes.c_int64(), ctypes.c_size_t()
    fake = ctypes.c_void_p(1 << 20)
    n0 = lib.tf_launch_count()
    assert lib.tf_bvh_build_sizes(100, None, ctypes.byref(ws)) != 0 and b"NULL pointer" in lib.tf_last_error()
    assert lib.tf_bvh_build_sizes(0, ctypes.byref(n_nodes), ctypes.byref(ws)) != 0 and b"empty mesh" in lib.tf_last_error()
    assert lib.tf_bvh_build_sizes(1 << 31, ctypes.byref(n_nodes), ctypes.byref(ws)) != 0 and b"2^31" in lib.tf_last_error()
    args = [fake, 300, fake, 100, fake, 1 << 30, fake, fake, fake, None]
    for i in (0, 2, 4, 6, 7, 8):
        a = list(args)
        a[i] = None
        assert lib.tf_bvh_build(*a) != 0 and b"NULL pointer" in lib.tf_last_error()
    assert lib.tf_bvh_build(*args[:3], 0, *args[4:]) != 0 and b"empty mesh" in lib.tf_last_error()
    assert lib.tf_bvh_build(*args[:3], 1 << 31, *args[4:]) != 0 and b"2^31" in lib.tf_last_error()
    a = list(args)
    a[6] = ctypes.c_void_p((1 << 20) + 4)
    assert lib.tf_bvh_build(*a) != 0 and b"aligned" in lib.tf_last_error()
    h = ctypes.c_void_p()
    assert lib.tf_bvh_create_from_device(fake, 10, None, fake, 20, None, ctypes.byref(h)) != 0
    assert b"NULL pointer" in lib.tf_last_error()
    assert lib.tf_bvh_create_from_device(fake, 10, fake, fake, 0, None, ctypes.byref(h)) != 0 and b"empty" in lib.tf_last_error()
    assert lib.tf_bvh_export(None, ctypes.byref(n_nodes), None, None, None, None) != 0 and b"NULL handle" in lib.tf_last_error()
    assert lib.tf_launch_count() == n0
