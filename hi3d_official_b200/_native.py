"""ctypes binding of libhi3d_b200.so (C ABI in include/hi3d_b200.h).

There is NO fallback: if the library cannot be loaded the import of any compute path raises, and every
entry point raises `Hi3dError` on a non-zero return code.  The library is built in-tree by `build.py`
(nvcc, sm_100a); on a box without nvcc the prebuilt .so that travelled with the snapshot is used.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

MAX_SEGS = 24
ROWS_PLAIN, ROWS_CONV2D, ROWS_TEMPORAL = 0, 1, 2
ACT_NONE, ACT_SILU, ACT_GEGLU = 0, 1, 2


class Hi3dError(RuntimeError):
    pass


class Seg(C.Structure):
    _fields_ = [("src", C.c_void_p), ("ld", C.c_int32), ("c_off", C.c_int32), ("C", C.c_int32),
                ("dy", C.c_int32), ("dx", C.c_int32), ("dt", C.c_int32)]


class GemmParams(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("mode", C.c_int32),
                ("Ho", C.c_int32), ("Wo", C.c_int32), ("Hs", C.c_int32), ("Ws", C.c_int32),
                ("stride", C.c_int32), ("ups", C.c_int32), ("T", C.c_int32),
                ("out_up", C.c_int32), ("out_py", C.c_int32), ("out_px", C.c_int32),
                ("Tin", C.c_int32), ("t_off", C.c_int32), ("nseg", C.c_int32),
                ("seg", Seg * MAX_SEGS),
                ("W", C.c_void_p), ("bias", C.c_void_p), ("rowbias", C.c_void_p),
                ("rb_div", C.c_int32), ("rb_mod", C.c_int32), ("rb_ld", C.c_int32), ("act", C.c_int32),
                ("residual", C.c_void_p), ("res_ld", C.c_int32),
                ("blend_x", C.c_void_p), ("blend_ld", C.c_int32), ("alpha", C.c_float),
                ("out", C.c_void_p), ("out_ld", C.c_int32),
                ("gn_stats", C.c_void_p), ("gn_unit", C.c_int32), ("gn_rows", C.c_int32)]


_lib = None

_SIGS = {
    "hi3d_abi_version": (C.c_int, []),
    "hi3d_last_error": (C.c_char_p, []),
    "hi3d_launch_count": (C.c_int64, []),
    "hi3d_device_info": (C.c_int, [C.POINTER(C.c_int)] * 4),
    "hi3d_gemm": (C.c_int, [C.POINTER(GemmParams), C.c_void_p]),
    "hi3d_gemm_tc5": (C.c_int, [C.POINTER(GemmParams), C.c_void_p]),
    "hi3d_gemm_tc5_set_pair_mode": (C.c_int, [C.c_int]),
    "hi3d_gemm_det": (C.c_int, [C.POINTER(GemmParams), C.c_void_p, C.c_int64, C.c_void_p]),
    "hi3d_gemm_tc5_det": (C.c_int, [C.POINTER(GemmParams), C.c_void_p, C.c_int64, C.c_void_p]),
    "hi3d_gemm_tc5_set_epilogue_warps": (C.c_int, [C.c_int]),
    "hi3d_groupnorm_ws_floats": (C.c_int64, [C.c_int]),
    "hi3d_groupnorm_silu": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p,
                                      C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hi3d_groupnorm_sums": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "hi3d_groupnorm_apply": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_int64, C.c_int64,
                                       C.c_void_p]),
    "hi3d_groupnorm_apply_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                             C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_float, C.c_int,
                                             C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "hi3d_groupnorm_unit_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "hi3d_groupnorm_group_sums": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p]),
    "hi3d_groupnorm_apply_halo": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_int64,
                                            C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_int64, C.c_int64,
                                            C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "hi3d_groupnorm_silu_det": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p,
                                          C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hi3d_groupnorm_sums_det": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "hi3d_groupnorm_group_sums_det": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                C.c_void_p, C.c_void_p]),
    "hi3d_groupnorm_unit_stats_det": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_int64, C.c_void_p]),
    "hi3d_groupnorm_partials_floats": (C.c_int64, [C.c_int, C.c_int64, C.c_int, C.c_int]),
    "hi3d_groupnorm_fold": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "hi3d_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p,
                                 C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "hi3d_attention_d64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "hi3d_attention_d64_tc5": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "hi3d_attention_d512_tc5": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "hi3d_attention_tc5_set_exp_emulation": (C.c_int, [C.c_int]),
    "hi3d_attention_tc5_set_variant": (C.c_int, [C.c_int]),
    "hi3d_attention_tc5_set_debug_buffer": (C.c_int, [C.c_void_p]),
    "hi3d_temporal_attention_d64": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                              C.c_void_p, C.c_void_p]),
    "hi3d_temporal_attention_d64_sharded": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int,
                                                      C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "hi3d_symm_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]),
    "hi3d_symm_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "hi3d_symm_close": (C.c_int, [C.c_void_p]),
    "hi3d_symm_free": (C.c_int, [C.c_void_p]),
    "hi3d_peer_xchg_bytes": (C.c_int64, [C.c_int]),
    "hi3d_peer_exchange": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "hi3d_softmax_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_void_p]),
    "hi3d_transpose": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "hi3d_timestep_embedding": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "hi3d_sampler_pre": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hi3d_sampler_post": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                    C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hi3d_sampler_lincomb4": (C.c_int, [C.c_void_p] * 9 + [C.c_int, C.c_int64, C.c_void_p]),
    "hi3d_renoise_blend": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int64,
                                     C.c_void_p]),
    "hi3d_nchw_to_nhwc": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                    C.c_void_p, C.c_void_p]),
    "hi3d_nhwc_to_nchw": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                    C.c_int, C.c_void_p]),
    "hi3d_gaussian_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_float, C.c_void_p, C.c_void_p]),
    "hi3d_pack_weight": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p]),
    "hi3d_pack_bias": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
}
EXPORTS = tuple(_SIGS)


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load (building first when nvcc + sources are newer) and type the C ABI.  Raises on any failure."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing:
        try:
            if not _build.is_fresh():
                _build.build()
        except Exception as e:  # no nvcc on this box: fall through to the prebuilt .so if there is one
            if not os.path.exists(path):
                raise Hi3dError(f"libhi3d_b200.so is missing and could not be built: {e}") from e
    if not os.path.exists(path):
        raise Hi3dError(f"{path} not found: run `python -m hi3d_official_b200.build` (needs nvcc)")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)   # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.hi3d_abi_version() != 2:
        raise Hi3dError("libhi3d_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().hi3d_last_error()
        raise Hi3dError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


_replayed = 0      # launches executed through CUDA-graph replays (the C counter only sees eager / capture-time calls)


def launch_count() -> int:
    return int(load().hi3d_launch_count()) + _replayed


def note_graph_replay(n_launches: int):
    """A CUDA graph holding `n_launches` of this library's kernels was replayed once."""
    global _replayed
    _replayed += int(n_launches)
