"""ctypes binding of libmimo_b200.so (the C ABI declared in include/mimo_b200.h).

Loading never needs a GPU (symbol checks run on CPU); every compute entry point fails loudly without an
sm_100 device — there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libmimo_b200.so"

F16, BF16 = 0, 1
ACT_NONE, ACT_SILU, ACT_GEGLU = 0, 1, 2


class MimoError(RuntimeError):
    pass


class Epilogue(C.Structure):
    _fields_ = [
        ("bias", C.c_void_p),
        ("rowvec", C.c_void_p),
        ("rows_per_group", C.c_int64),
        ("ld_rowvec", C.c_int64),
        ("residual", C.c_void_p),
        ("ld_res", C.c_int64),
        ("scale", C.c_float),
        ("act", C.c_int),
    ]


class GemmParams(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("lda", C.c_int64),
        ("a1", C.c_void_p), ("lda1", C.c_int64),
        ("w", C.c_void_p), ("ldw", C.c_int64),
        ("out", C.c_void_p), ("ldo", C.c_int64),
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("K1", C.c_int32),
        ("dtype", C.c_int32),
        ("ep", Epilogue),
    ]


class Conv3x3Params(C.Structure):
    _fields_ = [
        ("x0", C.c_void_p), ("c0", C.c_int32),
        ("x1", C.c_void_p), ("c1", C.c_int32),
        ("w", C.c_void_p),
        ("out", C.c_void_p), ("ldo", C.c_int64),
        ("n", C.c_int32), ("h", C.c_int32), ("w_", C.c_int32), ("cout", C.c_int32),
        ("dtype", C.c_int32),
        ("ep", Epilogue),
    ]


class GroupNormParams(C.Structure):
    _fields_ = [
        ("x0", C.c_void_p), ("c0", C.c_int32),
        ("x1", C.c_void_p), ("c1", C.c_int32),
        ("gamma", C.c_void_p), ("beta", C.c_void_p),
        ("out", C.c_void_p),
        ("stats", C.c_void_p),
        ("n", C.c_int32), ("hw", C.c_int32), ("groups", C.c_int32),
        ("eps", C.c_float),
        ("silu", C.c_int32),
        ("dtype", C.c_int32),
    ]


class AttnParams(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("ld_qkv", C.c_int64),
        ("bank_k", C.c_void_p), ("bank_v", C.c_void_p), ("ld_bank", C.c_int64),
        ("lb", C.c_int32), ("nb", C.c_int32),
        ("bank_index", C.c_void_p),
        ("out", C.c_void_p), ("ld_out", C.c_int64),
        ("n", C.c_int32), ("lq", C.c_int32), ("heads", C.c_int32), ("d", C.c_int32),
        ("scale", C.c_float),
        ("dtype", C.c_int32),
    ]


class AttnTemporalParams(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("ld_q", C.c_int64),
        ("k", C.c_void_p), ("v", C.c_void_p), ("ld_kv", C.c_int64),
        ("out", C.c_void_p), ("ld_out", C.c_int64),
        ("chunk_stride_rows", C.c_int64),
        ("batch", C.c_int32), ("q_frames", C.c_int32), ("kv_frames", C.c_int32), ("frames_per_chunk", C.c_int32),
        ("hw", C.c_int32), ("heads", C.c_int32), ("d", C.c_int32),
        ("scale", C.c_float),
        ("dtype", C.c_int32),
    ]


MAX_PEERS = 8


class ExchangeParams(C.Structure):
    _fields_ = [
        ("peer_src", C.c_void_p * MAX_PEERS), ("peer_ready", C.c_void_p * MAX_PEERS),
        ("ctl", C.c_void_p), ("dst", C.c_void_p), ("residual", C.c_void_p),
        ("mode", C.c_int32), ("G", C.c_int32), ("r", C.c_int32),
        ("b", C.c_int32), ("fl", C.c_int32), ("hw", C.c_int32), ("C", C.c_int32),
        ("dtype", C.c_int32), ("max_blocks", C.c_int32), ("timeout_ms", C.c_int32),
    ]


# every symbol include/mimo_b200.h declares: name -> (restype, argtypes)
_VP, _I32, _I64, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float
SYMBOLS = {
    "mimo_version": (C.c_char_p, []),
    "mimo_last_error": (C.c_char_p, []),
    "mimo_device_check": (C.c_int, [C.c_int]),
    "mimo_abi_sizeof": (C.c_int, [C.c_int]),
    "mimo_gemm": (C.c_int, [C.POINTER(GemmParams), _VP]),
    "mimo_gemm_geglu_granule": (C.c_int, [_I32]),
    "mimo_conv3x3": (C.c_int, [C.POINTER(Conv3x3Params), _VP]),
    "mimo_conv_up2x": (C.c_int, [C.POINTER(Conv3x3Params), _VP]),
    "mimo_im2col3x3": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I64, _I32, _VP]),
    "mimo_groupnorm": (C.c_int, [C.POINTER(GroupNormParams), _VP]),
    "mimo_groupnorm_workspace_bytes": (C.c_int64, [C.POINTER(GroupNormParams)]),
    "mimo_layernorm": (C.c_int, [_VP, _VP, _VP, _VP, _I64, _I32, _F, _VP, _I64, _I32, _I32, _I32, _VP]),
    "mimo_attn_spatial": (C.c_int, [C.POINTER(AttnParams), _VP]),
    "mimo_attn_temporal": (C.c_int, [C.POINTER(AttnTemporalParams), _VP]),
    "mimo_exchange": (C.c_int, [C.POINTER(ExchangeParams), _VP]),
    "mimo_peer_alloc": (C.c_int, [_I64, C.POINTER(C.c_void_p), C.c_char_p]),
    "mimo_peer_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "mimo_peer_close": (C.c_int, [_VP]),
    "mimo_peer_free": (C.c_int, [_VP]),
    "mimo_ncfhw_to_nhwc": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _VP]),
    "mimo_nhwc_to_ncfhw": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _VP]),
    "mimo_upsample2x": (C.c_int, [_VP, _VP, _I32, _I32, _I32, _I32, _I32, _VP]),
    "mimo_softmax_rows": (C.c_int, [_VP, _I64, _I32, _I64, _I32, _VP]),
    "mimo_add": (C.c_int, [_VP, _VP, _VP, _I64, _I32, _VP]),
    "mimo_silu": (C.c_int, [_VP, _VP, _I64, _I32, _VP]),
    "mimo_quick_gelu": (C.c_int, [_VP, _VP, _I64, _I32, _VP]),
    "mimo_composite_frame": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_double, _VP, _I64, _VP]),
    "mimo_cfg_ddim_step": (C.c_int, [_VP, _VP, _VP, _I64, _VP, _I64, _F, _F, _F, _F, _F, _I32, _VP]),
}
# test hook, not part of the public header
_DEBUG_SYMBOLS = {"mimo_debug_pdl": (C.c_int, [C.c_int]), "mimo_debug_force_bn": (C.c_int, [C.c_int]),
                  "mimo_debug_gemm_trace": (C.c_int, [C.c_void_p])}

_lib = None


def load() -> C.CDLL:
    """Load the library (building is build.py's / __graft_entry__.build()'s job, never done implicitly)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise MimoError(
            f"{LIB_PATH} is missing: run `python -m mimo_b200.build` (or __graft_entry__.build()). "
            "mimo_b200 has no CPU or PyTorch fallback."
        )
    lib = C.CDLL(os.fspath(LIB_PATH))
    for name, (res, args) in {**SYMBOLS, **_DEBUG_SYMBOLS}.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    for which, st in enumerate((Epilogue, GemmParams, Conv3x3Params, GroupNormParams, AttnParams, AttnTemporalParams,
                             ExchangeParams)):
        if lib.mimo_abi_sizeof(which) != C.sizeof(st):
            raise MimoError(f"ABI mismatch: {st.__name__} is {C.sizeof(st)} bytes in lib.py but "
                            f"{lib.mimo_abi_sizeof(which)} in {LIB_PATH.name}; rebuild the library")
    if os.environ.get("MIMO_B200_PDL") in ("0", "1"):  # A/B switch for programmatic dependent launch (default: off)
        lib.mimo_debug_pdl(int(os.environ["MIMO_B200_PDL"]))
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mimo_last_error().decode(errors="replace")
        raise MimoError(f"{what or 'mimo call'} failed (rc={rc}): {msg}")
