"""ctypes binding of libactionmesh_b200.so (the C ABI declared in include/actionmesh_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails the error is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libactionmesh_b200.so")

ABI_VERSION = 14

EXPORTS = [
    "amb_last_error", "amb_abi_version", "amb_device_info", "amb_cfg_euler_step", "amb_layernorm",
    "amb_cast_f32_bf16", "amb_patchify", "amb_timestep_embedding", "amb_alpha_rows", "amb_point_embedding",
    "amb_displacement_out", "amb_split3_bf16", "amb_softmax_split3", "amb_resize_h_u8", "amb_resize_v_normalize", "amb_alpha_stats", "amb_composite_crop_pad", "amb_nearest_neighbors", "amb_icp_workspace_bytes", "amb_icp_chamfer_grad", "amb_gradient_icp",
    "amb_transform_points", "amb_add_bias_rows", "amb_gemm_bf16", "amb_flash_attn_fwd", "amb_attn_small_f32", "amb_debug_set_attn_trace",
]


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("lda", C.c_int64),
        ("a2", C.c_void_p), ("lda2", C.c_int64), ("k_split", C.c_int32),
        ("w", C.c_void_p), ("ldw", C.c_int64),
        ("c", C.c_void_p), ("ldc", C.c_int64), ("c_fp32", C.c_int32),
        ("m", C.c_int32), ("n", C.c_int32), ("k", C.c_int32),
        ("bias", C.c_void_p),
        ("residual", C.c_void_p), ("ldr", C.c_int64), ("res_fp32", C.c_int32),
        ("act", C.c_int32),
        ("col_scale", C.c_void_p),
        ("grp_rows", C.c_int32), ("grp_stride", C.c_int32), ("row_off", C.c_int32),
        ("norm_cols", C.c_int32), ("norm_seg", C.c_int32),
        ("norm_w0", C.c_void_p), ("norm_w1", C.c_void_p), ("norm_eps", C.c_float),
        ("rope_cols", C.c_int32), ("rope_cos", C.c_void_p), ("rope_sin", C.c_void_p),
        ("rope_rows_per_pos", C.c_int32),
        ("c2", C.c_void_p), ("ldc2", C.c_int64),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("o", C.c_void_p),
        ("q_stride_b", C.c_int64), ("q_stride_h", C.c_int64), ("q_stride_s", C.c_int64),
        ("k_stride_b", C.c_int64), ("k_stride_h", C.c_int64), ("k_stride_s", C.c_int64),
        ("v_stride_b", C.c_int64), ("v_stride_h", C.c_int64), ("v_stride_s", C.c_int64),
        ("o_stride_b", C.c_int64), ("o_stride_h", C.c_int64), ("o_stride_s", C.c_int64),
        ("batch", C.c_int32), ("heads", C.c_int32), ("sq", C.c_int32), ("sk", C.c_int32), ("head_dim", C.c_int32),
        ("scale", C.c_float),
        ("kv_chunks", C.c_int32), ("sk_chunk", C.c_int32),
        ("k_chunk_stride", C.c_int64), ("v_chunk_stride", C.c_int64),
    ]


_lib = None


class AmbError(RuntimeError):
    pass


def load_library() -> C.CDLL:
    """Load the CUDA extension; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AmbError(
            f"{LIB_PATH} not found: the sm_100a CUDA extension has not been built. "
            "Run `python __graft_entry__.py` (there is no CPU fallback)."
        )
    lib = C.CDLL(LIB_PATH)
    lib.amb_last_error.restype = C.c_char_p
    lib.amb_abi_version.restype = C.c_int
    if lib.amb_abi_version() != ABI_VERSION:
        raise AmbError(f"ABI mismatch: library {lib.amb_abi_version()} != binding {ABI_VERSION}; rebuild")
    lib.amb_device_info.argtypes = [C.POINTER(C.c_int)] * 3
    lib.amb_cfg_euler_step.argtypes = [
        C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float), C.c_float, C.c_void_p, C.c_int, C.c_int64,
        C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
    ]
    lib.amb_layernorm.argtypes = [
        C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int,
        C.c_float, C.c_void_p,
    ]
    lib.amb_alpha_rows.argtypes = [C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
    lib.amb_point_embedding.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    lib.amb_displacement_out.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.amb_split3_bf16.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
    lib.amb_softmax_split3.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int64, C.c_void_p]
    lib.amb_resize_h_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.amb_resize_v_normalize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                           C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_void_p,
                                           C.c_void_p]
    lib.amb_alpha_stats.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.amb_composite_crop_pad.argtypes = [C.c_void_p] + [C.c_int] * 9 + [C.c_void_p, C.c_void_p]
    lib.amb_nearest_neighbors.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.amb_icp_workspace_bytes.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    lib.amb_icp_chamfer_grad.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.amb_gradient_icp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]
    lib.amb_transform_points.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.amb_patchify.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.amb_cast_f32_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.amb_timestep_embedding.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.amb_add_bias_rows.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
    lib.amb_gemm_bf16.argtypes = [C.POINTER(GemmArgs), C.c_void_p]
    lib.amb_flash_attn_fwd.argtypes = [C.POINTER(AttnArgs), C.c_void_p]
    lib.amb_debug_set_attn_trace.argtypes = [C.c_void_p]
    lib.amb_attn_small_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float,
                                       C.c_void_p, C.c_int64, C.c_void_p]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name != "amb_last_error":
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().amb_last_error().decode(errors="replace")
        raise AmbError(f"{what} failed (code {rc}): {msg}")
