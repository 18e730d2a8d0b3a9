"""ctypes binding of libpbg_b200.so (the C ABI in include/pbg.h).

This is the only way the Python host reaches the kernels; there is no fallback: if the shared
library is missing it is built with nvcc, and if that is impossible an ImportError-style
RuntimeError is raised.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

PBG_OK, PBG_ERR_INVALID, PBG_ERR_CUDA, PBG_ERR_NOT_LOADED, PBG_ERR_INDEX, PBG_ERR_UNSUPPORTED, PBG_ERR_NOMEM = range(7)
PREC_F32, PREC_BF16 = 0, 1
DT_F32, DT_BF16 = 0, 1
KERNEL_KINDS = ("gather", "g_l0", "g_l1", "g_l2", "d_l0", "d_l1", "other", "pass", "topk")

# every symbol include/pbg.h declares (tests check the .so exports exactly these)
SYMBOLS = (
    "pbg_abi_version", "pbg_create", "pbg_destroy", "pbg_last_error", "pbg_load_generator",
    "pbg_load_discriminator", "pbg_generator_forward", "pbg_generator_forward_gather",
    "pbg_discriminator_forward", "pbg_discriminator_score_triplets", "pbg_score_triplets",
    "pbg_score_triplets_host", "pbg_linear_bf16", "pbg_profile_enable", "pbg_profile_read", "pbg_debug_trace", "pbg_check_indices", "pbg_launch_count",
    "pbg_set_launch_width", "pbg_set_result_mirrors", "pbg_topk_prepare", "pbg_topk", "pbg_parse_index_rows", "pbg_format_f32_json", "pbg_format_i64_json",
    "pbg_reserve", "pbg_stage_triplets", "pbg_score_staged", "pbg_set_result_multicast", "pbg_topk_last_flagged", "pbg_score_triplets_host_packed", "pbg_score_staged_stage_next", "pbg_set_workspace_discard", "pbg_last_pass_sm_clock",
    "pbg_draw_latents", "pbg_set_latent_stream", "pbg_get_latent_stream", "pbg_score_triplets_host_ids",
)


class PbgDims(C.Structure):
    _fields_ = [("embed_dim", C.c_int32), ("noise_dim", C.c_int32), ("g_hidden", C.c_int32),
                ("d_hidden", C.c_int32), ("device", C.c_int32), ("leaky_slope", C.c_float)]


class PbgError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libpbg_b200 status {status}: {message}")
        self.status = status


_lib = None


def lib_path() -> Path:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """dlopen the in-tree library (building it first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    import os
    override = os.environ.get("PBG_LIB_PATH")     # an A/B build of the same sources (pbg.build --variant), never a fallback
    path = Path(override) if override else _build.build()
    lib = C.CDLL(str(path))
    vp, i64, i32, sz, u64 = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_uint64
    sig = {
        "pbg_abi_version": (C.c_int, []),
        "pbg_create": (C.c_int, [C.POINTER(vp), C.POINTER(PbgDims)]),
        "pbg_destroy": (None, [vp]),
        "pbg_last_error": (C.c_char_p, [vp]),
        "pbg_load_generator": (C.c_int, [vp, vp, sz]),
        "pbg_load_discriminator": (C.c_int, [vp, vp, sz]),
        "pbg_generator_forward": (C.c_int, [vp, vp, vp, vp, vp, i64, i32, i32, vp]),
        "pbg_generator_forward_gather": (C.c_int, [vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, vp, i64, i32, i32, vp]),
        "pbg_discriminator_forward": (C.c_int, [vp, vp, vp, vp, vp, vp, i64, i32, vp]),
        "pbg_discriminator_score_triplets": (C.c_int, [vp, vp, i64, vp, i64, vp, vp, vp, i64, i32, vp]),
        "pbg_score_triplets": (C.c_int, [vp, vp, i64, vp, i64, vp, vp, vp, i32, vp, vp, vp, i64, i32, vp]),
        "pbg_score_triplets_host": (C.c_int, [vp, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, i64, i32]),
        "pbg_linear_bf16": (C.c_int, [vp, i32, i32, vp, vp, i64, vp]),
        "pbg_profile_enable": (C.c_int, [vp, i32]),
        "pbg_profile_read": (C.c_int, [vp, vp, vp]),
        "pbg_debug_trace": (C.c_int, [vp, i32, vp, i64]),
        "pbg_check_indices": (C.c_int, [vp, vp]),
        "pbg_launch_count": (i64, [vp]),
        "pbg_set_launch_width": (C.c_int, [vp, i32]),
        "pbg_set_workspace_discard": (C.c_int, [vp, i32]),
        "pbg_last_pass_sm_clock": (C.c_int, [vp, vp, C.POINTER(C.c_double)]),
        "pbg_set_result_mirrors": (C.c_int, [vp, i32, vp, vp, vp, vp]),
        "pbg_topk_prepare": (C.c_int, [vp, vp, i64, vp]),
        "pbg_topk": (C.c_int, [vp, vp, i64, i32, vp, vp, vp]),
        "pbg_parse_index_rows": (i64, [C.c_char_p, sz, i32, vp, sz]),
        "pbg_format_f32_json": (i64, [vp, sz, i32, i32, i32, vp, sz]),
        "pbg_format_i64_json": (i64, [vp, sz, i32, i32, i32, vp, sz]),
        "pbg_reserve": (C.c_int, [vp, i64, i32, i32]),
        "pbg_stage_triplets": (C.c_int, [vp, i32, vp, i64, vp, i64, vp, vp, i64, i32, i32, vp]),
        "pbg_score_staged": (C.c_int, [vp, i32, vp, i32, vp, vp, vp, vp]),
        "pbg_set_result_multicast": (C.c_int, [vp, vp, vp, vp, vp]),
        "pbg_topk_last_flagged": (i64, [vp, vp]),
        "pbg_score_triplets_host_packed": (C.c_int, [vp, vp, i64, vp, i64, vp, vp, i64, i32]),
        "pbg_score_staged_stage_next": (C.c_int, [vp, i32, vp, i32, vp, vp, vp, vp, i64, vp, i64, vp, vp, i64, vp]),
        "pbg_draw_latents": (C.c_int, [vp, u64, u64, i64, i64, i64, vp, C.POINTER(u64), vp]),
        "pbg_set_latent_stream": (C.c_int, [vp, i32, u64, u64]),
        "pbg_get_latent_stream": (C.c_int, [vp, C.POINTER(u64), C.POINTER(u64), vp]),
        "pbg_score_triplets_host_ids": (C.c_int, [vp, vp, i64, vp, i64, vp, vp, i64, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def last_error(handle) -> str:
    msg = load().pbg_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, handle=None) -> None:
    if status == PBG_OK:
        return
    msg = last_error(handle)
    if status == PBG_ERR_INDEX:
        # same exception type as the reference's `self.node_emb[heads]` (pro_b_gan_infer.py:139)
        raise IndexError(msg or "index out of range in embedding gather")
    raise PbgError(status, msg)
