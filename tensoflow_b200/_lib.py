"""ctypes binding of libtensoflow_b200.so (declared in include/tensoflow_b200.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is
raised.  The library is built in-tree by `python -m tensoflow_b200.build`.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

# TENSOFLOW_B200_LIB: explicit path of the shared library (deployments that keep it outside the package directory;
# scripts/stencil_phase_probe.py points it at the experiment build)
_LIB_PATH = Path(os.environ.get("TENSOFLOW_B200_LIB") or Path(__file__).resolve().parent / "libtensoflow_b200.so")
_lib = None


class VMField(C.Structure):
    _fields_ = [
        ("plane", C.c_void_p * 3), ("plane_mip", C.c_void_p * 3),
        ("line", C.c_void_p * 3), ("line_mip", C.c_void_p * 3),
        ("plane_h", C.c_int32 * 3), ("plane_w", C.c_int32 * 3), ("line_g", C.c_int32 * 3),
        ("n_comp", C.c_int32), ("n_levels", C.c_int32),
        ("aabb_min", C.c_float * 3), ("aabb_max", C.c_float * 3),
    ]


class VMMut(C.Structure):
    _fields_ = [("plane", C.c_void_p * 3), ("plane_mip", C.c_void_p * 3),
                ("line", C.c_void_p * 3), ("line_mip", C.c_void_p * 3)]


class SdfMlp(C.Structure):
    _fields_ = [("W0", C.c_void_p), ("b0", C.c_void_p), ("W1", C.c_void_p), ("b1", C.c_void_p),
                ("hidden", C.c_int32), ("app_dim", C.c_int32)]


class SdfMlpGrad(C.Structure):
    _fields_ = [("W0", C.c_void_p), ("b0", C.c_void_p), ("W1", C.c_void_p), ("b1", C.c_void_p)]


_P = C.c_void_p
_SIGNATURES = {
    "tf_abi_version": (C.c_int, []),
    "tf_last_error": (C.c_char_p, []),
    "tf_launch_count": (C.c_longlong, []),
    "tf_vm_build_mips": (C.c_int, [C.POINTER(VMField), C.POINTER(VMMut), _P]),
    "tf_vm_fold_mip_grads": (C.c_int, [C.POINTER(VMField), C.POINTER(VMMut), _P]),
    "tf_vm_feature_fwd": (C.c_int, [C.POINTER(VMField), _P, _P, C.c_int64, _P, _P]),
    "tf_vm_feature_bwd": (C.c_int, [C.POINTER(VMField), _P, _P, C.c_int64, _P, C.POINTER(VMMut), _P]),
    "tf_sdf_stencil_fwd_workspace": (C.c_size_t, [C.POINTER(VMField), C.POINTER(SdfMlp), C.c_int64, C.c_int32]),
    "tf_sdf_stencil_fwd": (C.c_int, [C.POINTER(VMField), C.POINTER(SdfMlp), _P, _P, C.c_int64,
                                     C.POINTER(C.c_float), _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "tf_sdf_only_fwd": (C.c_int, [C.POINTER(VMField), C.POINTER(SdfMlp), _P, _P, C.c_int64, _P, _P,
                                  C.c_size_t, _P]),
    "tf_sdf_point_fwd": (C.c_int, [C.POINTER(VMField), C.POINTER(SdfMlp), _P, _P, C.c_int64, _P, _P, _P, C.c_size_t, _P]),
    "tf_sdf_stencil_bwd_workspace": (C.c_size_t, [C.POINTER(VMField), C.POINTER(SdfMlp), C.c_int64]),
    "tf_sdf_stencil_bwd": (C.c_int, [C.POINTER(VMField), C.POINTER(SdfMlp), _P, _P, C.c_int64,
                                     C.POINTER(C.c_float), _P, _P, _P, _P, _P, C.POINTER(VMMut),
                                     C.POINTER(SdfMlpGrad), _P, C.c_size_t, _P]),
    "tf_sdf_stencil_fwd_hidden_offset": (C.c_size_t, [C.POINTER(VMField), C.POINTER(SdfMlp)]),
    "tf_sdf_stencil_bwd_kept": (C.c_int, [C.POINTER(VMField), C.POINTER(SdfMlp), _P, _P, C.c_int64,
                                          C.POINTER(C.c_float), _P, _P, _P, _P, _P, _P, C.POINTER(VMMut),
                                          C.POINTER(SdfMlpGrad), _P, C.c_size_t, _P]),
    "tf_neus_composite_fwd": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, _P, C.c_float, _P, C.c_int32,
                                        _P, _P, _P, _P, _P]),
    "tf_neus_composite_bwd": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, _P, C.c_float, _P, C.c_int32,
                                        _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_iso_count": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P]),
    "tf_iso_vertices": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P, _P]),
    "tf_iso_triangles": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, _P, _P]),
}

# later sections of the ABI (small MLP layers, flow sampler, MC shading, BVH)
_OPTIONAL_SIGNATURES = {
    "tf_linear_workspace": (C.c_size_t, [C.c_int32, C.c_int32]),
    "tf_linear_fwd": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, _P, _P, C.c_size_t, _P]),
    "tf_linear_bwd": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                _P, _P, _P, _P, C.c_size_t, _P]),
    "tf_pwquad_fwd": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, _P, _P]),
    "tf_pwquad_bwd": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P, _P]),
    "tf_bvh_create": (C.c_int, [_P, C.c_int64, _P, C.c_int64, C.POINTER(C.c_void_p)]),
    "tf_bvh_destroy": (None, [_P]),
    "tf_bvh_trace": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "tf_mc_directions": (C.c_int, [C.c_int32, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P]),
    "tf_cube_light_fwd": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int64, _P, _P]),
    "tf_cube_light_bwd": (C.c_int, [C.c_int32, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "tf_mc_estimate_fwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, C.c_int32, _P, _P,
                                     _P, _P]),
    "tf_mc_estimate_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, C.c_int32, _P, _P,
                                     _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_flow_block_fwd": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, C.c_float, C.c_float, C.c_int32, C.c_int32,
                                    C.c_int64, _P, _P, _P, _P, _P]),
    "tf_flow_block_uses_tensor_cores": (C.c_int, []),
    "tf_flow_block_bwd": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, C.c_float, C.c_float, C.c_int32, C.c_int64,
                                    _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_shader_encode_fwd": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_shader_encode_bwd": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_shader_combine_fwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P]),
    "tf_shader_combine_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_hit_encode": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, C.c_int32, _P, _P]),
    "tf_csr_spmm3_fwd": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P]),
    "tf_csr_spmm3_bwd": (C.c_int, [_P, _P, _P, _P, C.c_int32, _P, _P]),
    "tf_sampler_init": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(C.c_float), C.c_float, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "tf_sampler_upsample": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, C.c_int32, _P, C.c_float, C.c_float, C.c_int32,
                                      C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "tf_sampler_finalize": (C.c_int, [_P, _P, _P, C.POINTER(C.c_float), C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "tf_probe_init": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "tf_probe_weights": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "tf_alpha_mask_sample": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), _P, C.c_int64, _P, _P]),
    "tf_gauss_residual_fwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.c_int32, C.c_int32, _P, _P, _P]),
    "tf_gauss_residual_bwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.c_int32, C.c_int32, _P, _P, _P]),
    "tf_tv_fwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "tf_tv_bwd": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, _P, _P, _P]),
    "tf_cube_sample_fwd": (C.c_int, [_P, _P, C.c_int32, _P, _P, C.c_int64, _P, _P]),
    "tf_cube_sample_bwd": (C.c_int, [_P, _P, C.c_int32, _P, _P, C.c_int64, _P, _P, _P, _P, _P]),
    "tf_occ_march_count": (C.c_int, [_P, _P, _P, C.c_int32, C.c_float, C.c_float, _P, _P, _P, _P, _P]),
    "tf_occ_march_write": (C.c_int, [_P, _P, _P, C.c_int32, C.c_float, C.c_float, _P, _P, _P, _P, _P, _P, _P, _P]),
    "tf_adam_step": (C.c_int, [C.c_int32, _P, _P, _P, _P, _P, _P, C.c_float, C.c_float, C.c_float, C.c_int32, _P]),
    "tf_kernel_timing_enable": (None, [C.c_int32]),
    "tf_kernel_timing_reset": (None, []),
    "tf_kernel_timing_read": (C.c_int, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "tf_xty_accumulate": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
}


def exported_symbols():
    """Names every include/*.h entry point must resolve to (used by the CPU tests)."""
    return sorted(list(_SIGNATURES) + list(_OPTIONAL_SIGNATURES))


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Load the shared library (no CUDA context needed)."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -m tensoflow_b200.build` "
            "(tensoflow_b200 has no CPU / PyTorch fallback)")
    lib = C.CDLL(str(_LIB_PATH))
    for name, (res, args) in {**_SIGNATURES, **_OPTIONAL_SIGNATURES}.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.tf_abi_version() != 1:
        raise RuntimeError("libtensoflow_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().tf_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL); enforces fp32/int32 CUDA contiguous."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("tensoflow_b200 kernels need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("internal error: non-contiguous tensor passed to the C ABI")
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count() -> int:
    """Kernels launched by libtensoflow_b200.so so far in this process."""
    return int(load().tf_launch_count())
