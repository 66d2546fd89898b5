"""ctypes binding of ``libneumesh_b200.so`` (the C ABI declared in ``include/neumesh_b200.h``).

There is no CPU implementation behind this module: if the shared library is missing or no CUDA device is present the
calls raise - nothing silently falls back to PyTorch or to the oracle.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libneumesh_b200.so")

MAX_LAYERS = 8


class FieldDesc(C.Structure):
    _fields_ = [
        ("D_density", C.c_int32), ("D_color", C.c_int32), ("W", C.c_int32), ("geometry_dim", C.c_int32),
        ("color_dim", C.c_int32), ("multires_d", C.c_int32), ("multires_fg", C.c_int32), ("multires_ft", C.c_int32),
        ("multires_view", C.c_int32), ("enable_nablas_input", C.c_int32), ("indicator_weight", C.c_float),
        ("s", C.c_float), ("geometry_features", C.c_void_p), ("color_features", C.c_void_p),
        ("indicator_vector", C.c_void_p), ("geo_v", C.c_void_p * MAX_LAYERS), ("geo_g", C.c_void_p * MAX_LAYERS),
        ("geo_b", C.c_void_p * MAX_LAYERS), ("col_w", C.c_void_p * MAX_LAYERS), ("col_b", C.c_void_p * MAX_LAYERS),
    ]


class RenderCfg(C.Structure):
    _fields_ = [
        ("obj_bounding_radius", C.c_float), ("N_samples", C.c_int32), ("N_importance", C.c_int32),
        ("N_upsample_iters", C.c_int32), ("bounded_near_far", C.c_int32), ("calc_normal", C.c_int32),
        ("white_bkgd", C.c_int32), ("use_near_bypass", C.c_int32), ("near_bypass", C.c_float),
        ("use_far_bypass", C.c_int32), ("far_bypass", C.c_float), ("normalize_dirs", C.c_int32),
        ("skip_dead_samples", C.c_int32), ("sampling_only", C.c_int32), ("perturb_u", C.c_void_p),
    ]


class RenderDetail(C.Structure):
    _fields_ = [("d_all", C.c_void_p), ("implicit_surface", C.c_void_p), ("implicit_nablas", C.c_void_p),
                ("radiance", C.c_void_p), ("sdf_mid", C.c_void_p), ("near_far", C.c_void_p)]


_lib = None

# every symbol include/neumesh_b200.h declares: (restype, argtypes)
_P, _I64, _I32, _F = C.c_void_p, C.c_int64, C.c_int32, C.c_float
SIGNATURES = {
    "nmb_last_error": (C.c_char_p, []),
    "nmb_version": (C.c_int, []),
    "nmb_launch_count": (_I64, []),
    "nmb_profile_enable": (None, [C.c_int]),
    "nmb_profile_collect": (C.c_int, [C.POINTER(C.c_double), C.POINTER(_I64), C.POINTER(_I64), C.c_int]),
    "nmb_grid_create": (C.c_int, [_P, _I64, _P, C.POINTER(_P)]),
    "nmb_grid_destroy": (None, [_P]),
    "nmb_grid_num_vertices": (_I64, [_P]),
    "nmb_grid_order": (_P, [_P]),
    "nmb_knn": (C.c_int, [_P, _P, _I64, C.c_int, _F, _P, _P, _P]),
    "nmb_mesh_distance": (C.c_int, [_P, _P, _F, _P, _I64, _P, _P, _P, _P, _P]),
    "nmb_field_create": (C.c_int, [_P, C.POINTER(FieldDesc), C.c_int, _P, C.POINTER(_P)]),
    "nmb_field_destroy": (None, [_P]),
    "nmb_field_update": (C.c_int, [_P, C.POINTER(FieldDesc), _P]),
    "nmb_field_shell_grid": (C.c_int, [_P, _P, C.POINTER(_I32), C.POINTER(_F), _P]),
    "nmb_field_sdf": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "nmb_field_forward": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P]),
    "nmb_field_forward_ex": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "nmb_field_color": (C.c_int, [_P, _P, _I64, _P, _P, _P, _P, _P, _I64, _P, _P]),
    "nmb_render_workspace_bytes": (_I64, [C.POINTER(RenderCfg), _I64]),
    "nmb_render": (C.c_int, [_P, C.POINTER(RenderCfg), _P, _P, _I64, _I64, _P, _P, _P, _P, C.POINTER(RenderDetail),
                             _P, _I64, _P]),
    "nmb_upsample_step": (C.c_int, [_P, _P, _I64, _I32, _I32, _F, _P, _P, _P]),
    "nmb_first_crossing": (C.c_int, [_P, _I64, _I32, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "nmb_pack_bgr8": (C.c_int, [_P, _I64, _P, _P]),
    "nmb_vertex_normals": (C.c_int, [_P, _I64, _P, _I64, _P, _P]),
    "nmb_get_rays": (C.c_int, [C.POINTER(_F), C.POINTER(_F), _I32, _I32, _P, _P, _P]),
    "nmb_mc_workspace_bytes": (_I64, [_I64, _I64, _I64]),
    "nmb_mc_count": (C.c_int, [_P, _I64, _I64, _I64, C.c_double, _P, _I64, C.POINTER(_I64), C.POINTER(_I64), _P]),
    "nmb_mc_emit": (C.c_int, [_P, _I64, _I64, _I64, C.c_double, _P, _I64, _P, _P, _P]),
    # training-path primitives (csrc/train.cu); the nmb_tr_inputs struct is bound in train_ops.TrInputs
    "nmb_tr_gemm": (C.c_int, [_P, _I64, C.c_int, _P, _I64, C.c_int, _P, _I64, _I64, _I64, _I64, _P, C.c_int, _P, _I64,
                              C.c_int, _P]),
    "nmb_tr_prep": (C.c_int, [_P, _P]),
    "nmb_tr_softplus_fwd": (C.c_int, [_P, _P, _P, _P, _I64, _P]),
    "nmb_tr_softplus_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _P]),
    "nmb_tr_geo_out_fwd": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P, _I64, _P]),
    "nmb_tr_color_out_fwd": (C.c_int, [_P, _P, _P, _I64, _I32, _P, _P]),
    "nmb_tr_color_out_bwd": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P]),
    "nmb_tr_colsum": (C.c_int, [_P, _I64, _I64, _I64, _P, _P]),
    "nmb_tr_geo_out_bwd": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _P, _I64, _I32, _P, _P, _P, _P, _P, _P]),
    "nmb_tr_input_bwd": (C.c_int, [_P, _P, _I64, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _P]),
}


def lib():
    """The loaded library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "neumesh_b200: %s not found - build it with `python -m neumesh_b200.build` "
                "(there is no CPU / PyTorch fallback for the CUDA kernels)" % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError("neumesh_b200: %s (code %d)" % (lib().nmb_last_error().decode(), rc))


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError("neumesh_b200.%s needs CUDA tensors: the kernels have no CPU implementation" % what)


def launch_count() -> int:
    return int(lib().nmb_launch_count())


PROFILE_CLASSES = ("knn", "bound_scan", "geo", "geo_jvp", "color", "sampler", "knn_list")


def profile_enable(on: bool):
    lib().nmb_profile_enable(1 if on else 0)


def profile_collect():
    """-> {class: {"ms": float, "launches": int, "points": int}} since the last collect (synchronises)."""
    n = len(PROFILE_CLASSES)
    ms = (C.c_double * n)()
    la = (C.c_int64 * n)()
    un = (C.c_int64 * n)()
    lib().nmb_profile_collect(ms, la, un, n)
    return {k: {"ms": ms[i], "launches": int(la[i]), "points": int(un[i])} for i, k in enumerate(PROFILE_CLASSES)}
