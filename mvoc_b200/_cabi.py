"""ctypes binding of the C-ABI library ``libmvoc_b200.so`` (see include/mvoc_b200.h).

The library is the product: there is no Python/torch fallback for any of its
entry points.  Importing this module never compiles anything; ``load()`` raises
``MvocLibraryError`` when the shared object has not been built
(``python -c "import __graft_entry__ as g; g.build()"`` or ``make``).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_void_p

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libmvoc_b200.so")

MVOC_BF16, MVOC_F16, MVOC_F32 = 0, 1, 2
MVOC_MASK_U8, MVOC_MASK_F32 = 0, 1
MVOC_MAX_OBJECTS = 8
MVOC_EXCHANGE_WAIT_FUSED = 1 << 30


class MvocLibraryError(RuntimeError):
    """The CUDA extension is missing or does not match include/mvoc_b200.h."""


class MvocError(RuntimeError):
    """A C-ABI call returned a negative status (text from mvoc_last_error)."""


# name -> (restype, argtypes); mirrors include/mvoc_b200.h declaration by declaration
SIGNATURES = {
    "mvoc_version": (c_char_p, []),
    "mvoc_last_error": (c_char_p, []),
    "mvoc_device_check": (c_int, [c_int]),
    "mvoc_attn_fwd": (
        c_int,
        [c_void_p] * 4 + [c_int] * 5 + [c_int64] * 12 + [c_float, c_int, c_int, c_void_p],
    ),
    "mvoc_attn_causal_fwd": (
        c_int, [c_void_p] * 4 + [c_int] * 5 + [c_int64] * 12 + [c_float, c_int, c_void_p]),
    "mvoc_attn_fwd_trace": (
        c_int, [c_void_p] * 4 + [c_int] * 5 + [ctypes.POINTER(c_int64), c_int, c_float, c_int, c_int, c_void_p, c_void_p]),
    "mvoc_attn_d512_fwd": (
        c_int, [c_void_p] * 4 + [c_int] * 3 + [c_int64] * 8 + [c_float, c_int, c_void_p]),
    "mvoc_attn_d80_fwd": (
        c_int, [c_void_p] * 4 + [c_int] * 5 + [c_int64] * 12 + [c_float, c_int, c_void_p]),
    "mvoc_attn_temporal_fwd": (
        c_int,
        [c_void_p] * 4 + [c_int64, c_int, c_int, c_int] + [c_int64] * 12 + [c_float, c_int, c_void_p],
    ),
    "mvoc_attn_temporal_strided_fwd": (
        c_int,
        [c_void_p] * 4 + [c_int64, c_int64, c_int, c_int, c_int, ctypes.POINTER(c_int64), c_float, c_int, c_void_p],
    ),
    "mvoc_groupnorm_nhwc_partial_count": (c_int64, [c_int64, c_int]),
    "mvoc_groupnorm_nhwc_geometry": (
        c_int, [c_int64, c_int, c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int64)]),
    "mvoc_groupnorm_nhwc_stats": (
        c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "mvoc_groupnorm_nhwc_finalize": (
        c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "mvoc_groupnorm_nhwc_apply": (
        c_int, [c_void_p] * 6 + [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "mvoc_geglu": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "mvoc_gemm_plan": (c_int, [c_int64, c_int64, c_int, c_int, c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int),
                               ctypes.POINTER(c_int)]),
    "mvoc_upsample_nearest2x_nhwc": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "mvoc_concat_lastdim": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]),
    "mvoc_layernorm": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_float, c_int, c_void_p]),
    "mvoc_qk_blend": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_int, c_int, c_void_p],
    ),
    "mvoc_attn_pair_fwd": (
        c_int,
        [c_void_p] * 4 + [c_int] * 5 + [c_int64] * 12 + [c_int, c_float, c_int, c_int, c_void_p],
    ),
    "mvoc_qk_blend_strided": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    ),
    "mvoc_attn_inject_fwd": (
        c_int,
        [c_void_p] * 4 + [c_int64] * 4 + [c_int, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int,
                                          c_float, c_int, c_int, c_void_p],
    ),
    "mvoc_feature_blend": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_int, c_void_p],
    ),
    "mvoc_groupnorm_workspace_bytes": (c_int64, [c_int64, c_int]),
    "mvoc_groupnorm_silu": (
        c_int,
        [c_void_p] * 4 + [c_int64, c_int, c_int64, c_int, c_int, c_float, c_int, c_int, c_void_p, c_void_p],
    ),
    "mvoc_conv3x3_nhwc": (
        c_int, [c_void_p] * 6 + [c_int, c_void_p] + [c_int] * 5 + [c_int, c_int, c_void_p]),
    "mvoc_conv3x3_s2_nhwc": (c_int, [c_void_p] * 4 + [c_int] * 9 + [c_void_p]),
    "mvoc_temporal_conv3": (
        c_int, [c_void_p] * 5 + [c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "mvoc_linear": (
        c_int, [c_void_p] * 5 + [c_int64, c_int, c_int, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "mvoc_linear_geglu": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "mvoc_linear_gelu": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_int64, c_int64, c_int, c_int, c_void_p]),
    "mvoc_exchange_header_bytes": (c_int64, []),
    "mvoc_exchange_max_sites": (c_int, []),
    "mvoc_exchange_arena_create": (c_int, [c_int64, ctypes.POINTER(c_void_p), c_void_p]),
    "mvoc_exchange_arena_open": (c_int, [c_void_p, ctypes.POINTER(c_void_p)]),
    "mvoc_exchange_arena_close": (c_int, [c_void_p]),
    "mvoc_exchange_arena_destroy": (c_int, [c_void_p]),
    "mvoc_exchange_to_pixel_shards": (
        c_int, [c_void_p, ctypes.POINTER(c_void_p), c_int64, c_int, c_int, c_int, c_int, c_int64, c_int, c_int, c_int,
                c_void_p]),
    "mvoc_exchange_to_frame_shards": (
        c_int, [c_void_p, ctypes.POINTER(c_void_p), c_int64, c_int, c_int, c_int, c_int, c_int64, c_int, c_int, c_int,
                c_void_p]),
    "mvoc_exchange_allgather": (
        c_int, [c_void_p, c_int64, ctypes.POINTER(c_void_p), c_int64, c_int, c_int, c_int, c_void_p]),
    "mvoc_exchange_wait": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "mvoc_latent_composite": (
        c_int,
        [c_void_p] * 5 + [c_int, c_int64, c_int64, c_float, c_int, c_int, c_int, c_int, c_void_p],
    ),
    "mvoc_cfg_ddim_step": (
        c_int,
        [c_void_p] * 3 + [c_int64, c_float, c_double, c_double, c_int, c_int, c_void_p],
    ),
    "mvoc_ddim_inverse_step": (
        c_int,
        [c_void_p] * 3 + [c_int64, c_float, c_double, c_double, c_int, c_int, c_void_p],
    ),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library once and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MvocLibraryError(
            f"{LIB_PATH} not found: the CUDA extension has not been built. "
            "Run `make` (or __graft_entry__.build()) in the repo root; there is no CPU fallback."
        )
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # missing libcudart etc.
        raise MvocLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise MvocLibraryError(f"{LIB_PATH} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().mvoc_last_error().decode("utf-8", "replace")
        raise MvocError(f"{what} failed with status {status}: {msg}")


def version() -> str:
    return load().mvoc_version().decode()
