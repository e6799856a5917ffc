"""ctypes binding of libttb200.so (the C ABI in include/ttb200.h).

The library is the product; this module only declares signatures.  There is no fallback:
if the shared object is missing or no B200 is visible, using the package raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

# TTB_LIB: file name (inside the package) of an experimental build of the same sources, for A/B runs (scripts/build_variant.sh)
LIB_PATH = Path(__file__).resolve().parent / os.environ.get("TTB_LIB", "libttb200.so")

ABI_VERSION = 8
PRECISION = {"fp32": 0, "bf16": 1}
ERR_REF_INDEX, ERR_REF_SHAPE, ERR_REF_ASSERT = 10, 11, 12


class ModelDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "src_vocab_size", "tgt_vocab_size", "embedding_dim", "feedforward_dim", "num_encoder_layers",
        "num_decoder_layers", "num_heads", "src_pad_token_idx", "tgt_pad_token_idx", "precision", "max_positions")]


class GenerateStats(C.Structure):
    _fields_ = [("model_calls", C.c_int32), ("accepted_tokens", C.c_int32), ("produced_tokens", C.c_int32),
                ("unfinished", C.c_int32), ("error", C.c_int32), ("gpu_launches", C.c_int32),
                ("gpu_ms", C.c_float), ("reserved", C.c_float)]


# name -> (restype, argtypes); kept in one table so the CPU test-suite can check that the library
# exports every symbol the header declares.
SIGNATURES = {
    "ttb_abi_version": (C.c_int, []),
    "ttb_last_error": (C.c_char_p, []),
    "ttb_device_check": (C.c_int, [C.c_int]),
    "ttb_engine_create": (C.c_int, [C.POINTER(ModelDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "ttb_engine_destroy": (None, [C.c_void_p]),
    "ttb_engine_set_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "ttb_engine_finalize": (C.c_int, [C.c_void_p]),
    "ttb_make_drafts": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "ttb_encode_src": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "ttb_decode_tgt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                 C.c_void_p, C.c_void_p]),
    "ttb_greedy_speculative_generate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                  C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                  C.c_void_p, C.c_void_p, C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_greedy_speculative_generate_batches": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int32] * 9 +
                                                [C.c_void_p, C.c_void_p, C.POINTER(GenerateStats), C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_greedy_generate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_void_p, C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_greedy_generate_batches": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int32] * 5 +
                                    [C.c_void_p, C.POINTER(GenerateStats), C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_beam_search_generate":(C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 7 +
                                 [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_beam_search_generate_batches": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int32] * 6 +
                                         [C.c_void_p, C.c_void_p, C.POINTER(GenerateStats), C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_beam_speculative_generate": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 12 +
                                      [C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_beam_speculative_generate_batches": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int32] * 11 +
                                              [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(GenerateStats), C.POINTER(GenerateStats),
                                               C.c_void_p]),
    "ttb_sample_generate": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int32] * 4 + [C.c_float, C.c_int32, C.c_uint64] + [C.c_int32] * 3 +
                            [C.c_void_p, C.POINTER(GenerateStats), C.c_void_p]),
    "ttb_score_targets": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ttb_engine_get_draft_history": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "ttb_kernel_class_count": (C.c_int, []),
    "ttb_kernel_class_name": (C.c_char_p, [C.c_int32]),
    "ttb_engine_set_profiling": (C.c_int, [C.c_void_p, C.c_uint32]),
    "ttb_engine_get_profile": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ttb_engine_get_history": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_int32]),
    "ttb_gemm": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                           C.c_int32, C.c_void_p]),
    "ttb_gemm_bf16_out": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
}

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libttb200.so (built in-tree by `translation_transformer_b200/build.py`)."""
    global _lib
    if _lib is not None:
        return _lib
    import torch  # noqa: F401  (loads the CUDA runtime the library links against)
    if not LIB_PATH.exists():
        raise LibraryMissing(
            f"{LIB_PATH} not found: build it with `python -m translation_transformer_b200.build` "
            "(there is no CPU or PyTorch fallback for the hot path)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ttb_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libttb200 ABI {lib.ttb_abi_version()} != binding ABI {ABI_VERSION}: rebuild the library")
    _lib = lib
    return lib


def last_error() -> str:
    return load().ttb_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    msg = last_error()
    if rc == ERR_REF_INDEX:
        raise RuntimeError(msg)          # the reference raises RuntimeError (scatter out of bounds)
    if rc == ERR_REF_SHAPE:
        raise RuntimeError(msg)          # the reference raises RuntimeError (shape mismatch)
    if rc == ERR_REF_ASSERT:
        raise AssertionError(msg)        # the reference asserts (topk_in_each_group)
    if rc == 2 and ("must be" in msg or "must not" in msg):
        raise AssertionError(msg)        # argument checks the reference states as `assert`
    raise RuntimeError(f"{what} failed (code {rc}): {msg}")
