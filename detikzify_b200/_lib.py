"""
ctypes binding of ``libdtk_b200.so`` (the C ABI in ``include/detikzify_b200.h``).

The product path has NO CPU fallback: if the library is missing or a CUDA device is absent the
engine raises — nothing here routes to PyTorch ops or to the test oracle.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "csrc" / "libdtk_b200.so"


class DtkConfig(C.Structure):
    _fields_ = [
        ("hidden", C.c_int32), ("inter", C.c_int32), ("layers", C.c_int32), ("heads", C.c_int32),
        ("kv_heads", C.c_int32), ("head_dim", C.c_int32), ("vocab", C.c_int32), ("max_len", C.c_int32),
        ("rms_eps", C.c_float), ("rope_theta", C.c_float), ("rope_factor", C.c_float),
        ("rope_type", C.c_int32), ("rope_low_freq", C.c_float), ("rope_high_freq", C.c_float), ("rope_orig_max_pos", C.c_int32),
        ("v_hidden", C.c_int32), ("v_inter", C.c_int32), ("v_layers", C.c_int32), ("v_heads", C.c_int32),
        ("v_image", C.c_int32), ("v_patch", C.c_int32), ("v_act", C.c_int32), ("v_eps", C.c_float),
        ("concat", C.c_int32), ("image_token_id", C.c_int32), ("eos_token_id", C.c_int32),
        ("max_seqs", C.c_int32), ("max_batch", C.c_int32),
    ]


class DtkWeightInfo(C.Structure):
    _fields_ = [("name", C.c_char * 64), ("offset", C.c_uint64), ("nbytes", C.c_uint64),
                ("rows", C.c_int32), ("cols", C.c_int32)]


class DtkSampling(C.Structure):
    _fields_ = [("temperature", C.c_double), ("top_p", C.c_double), ("top_k", C.c_int32),
                ("do_sample", C.c_int32), ("bad_token", C.c_int32), ("begin_suppress_token", C.c_int32),
                ("seed", C.c_uint64)]


# every symbol include/detikzify_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "dtk_abi_version": (C.c_int, []),
    "dtk_weight_count": (C.c_int, [C.POINTER(DtkConfig)]),
    "dtk_weight_get": (C.c_int, [C.POINTER(DtkConfig), C.c_int, C.POINTER(DtkWeightInfo)]),
    "dtk_arena_bytes": (C.c_uint64, [C.POINTER(DtkConfig)]),
    "dtk_create": (C.c_int, [C.POINTER(DtkConfig), _P, C.c_uint64, C.c_int, C.POINTER(_P)]),
    "dtk_destroy": (C.c_int, [_P]),
    "dtk_last_error": (C.c_char_p, [_P]),
    "dtk_vit_encode": (C.c_int, [_P, _P, C.c_int, _P, _P, _P]),
    "dtk_project": (C.c_int, [_P, _P, C.c_int, _P, _P]),
    "dtk_image_preprocess": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, C.c_int, C.c_float,
                                       C.POINTER(C.c_float), C.POINTER(C.c_float), _P, _P, _P, _P]),
    "dtk_seq_alloc": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "dtk_seq_free": (C.c_int, [_P, C.c_int]),
    "dtk_seq_fork": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P]),
    "dtk_seq_share": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P]),
    "dtk_prefill": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, _P, _P]),
    "dtk_decode": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), _P, C.c_int, _P, _P]),
    "dtk_sample": (C.c_int, [_P, _P, C.c_int, C.POINTER(DtkSampling), C.POINTER(C.c_int),
                             C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), _P, _P, _P]),
    "dtk_gen_begin": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64), C.c_int,
                                C.POINTER(DtkSampling), C.POINTER(C.c_uint32), _P]),
    "dtk_gen_step": (C.c_int, [_P, _P]),
    "dtk_gen_wait": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int32)]),
    "dtk_gen_end": (C.c_int, [_P]),
    "dtk_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "dtk_get_option": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_int64)]),
    "dtk_decode_bytes": (C.c_uint64, [C.POINTER(DtkConfig), C.c_int]),
    "dtk_launch_count": (C.c_uint64, [_P]),
    "dtk_dbg_mega_times": (C.c_int, [_P, C.POINTER(C.c_longlong), C.c_int]),
    "dtk_dbg_mega_trace": (C.c_int, [_P, C.POINTER(C.c_longlong), C.c_int]),
    "dtk_dbg_gemm_impl": (C.c_int, [C.c_int]),
    "dtk_dbg_gemm": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "dtk_dbg_flash_attn": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_float, _P]),
    "dtk_dbg_flash_attn_ex": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "dtk_dbg_decode_attn": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_float, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "dtk_dbg_attn_tc": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "dtk_dbg_gemv": (C.c_int, [_P, _P, _P, C.c_float, C.c_int, C.c_int, C.c_int, _P, _P]),
}

_lib = None


def load_library(build_if_missing: bool = False) -> C.CDLL:
    """dlopen the in-tree library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if build_if_missing:
            from .build import build
            build()
        else:
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m detikzify_b200.build` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
    import os
    # dev aid for same-box A/B runs of two builds; the product path always loads the in-tree library
    lib = C.CDLL(os.environ.get("DTK_B200_LIB", str(LIB_PATH)))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dtk_abi_version() != 2:
        raise RuntimeError("libdtk_b200.so ABI version mismatch")
    _lib = lib
    return lib
