"""ctypes binding of libmw_b200.so (the C ABI declared in include/mw_b200.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

# MW_STORAGE_BF16=1 selects the bf16-storage A/B build (python -m manual_whisper_b200.build under the same variable)
_LIB_PATH = Path(__file__).resolve().parent / ("libmw_b200_bf16.so" if os.environ.get("MW_STORAGE_BF16") == "1" else "libmw_b200.so")
_lib = None

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_f32p = C.POINTER(C.c_float)


class GenOptionsC(C.Structure):
    _fields_ = [
        ("beam_size", C.c_int32), ("patience", C.c_float), ("length_penalty", C.c_float),
        ("max_length", C.c_int32),
        ("n_suppress", C.c_int32), ("h_suppress", c_i32p),
        ("n_suppress_begin", C.c_int32), ("h_suppress_begin", c_i32p),
        ("eot", C.c_int32), ("timestamp_begin", C.c_int32), ("no_timestamps", C.c_int32),
        ("with_timestamps", C.c_int32), ("max_initial_timestamp_index", C.c_int32),
        ("num_hypotheses", C.c_int32), ("forced_eot_len", C.c_int32),
    ]


class ModelConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_mels", "d_model", "n_heads", "enc_layers", "dec_layers", "ffn", "vocab",
        "n_audio_ctx", "n_text_ctx", "max_batch", "max_beam", "device")]


class W2vConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_layers", "d_model", "n_heads", "ffn", "vocab", "conv_dim", "pos_kernel", "pos_groups", "max_batch", "max_samples",
        "device", "variant")]


class WeightTableC(C.Structure):
    _fields_ = [("n", C.c_int32), ("ptrs", C.POINTER(C.c_void_p))]


# name -> (restype, argtypes).  Every symbol include/mw_b200.h declares is listed here;
# tests/test_abi.py checks the library exports each of them.
SIGNATURES = {
    "mw_abi_version": (C.c_int, []),
    "mw_storage_dtype": (C.c_int, []),
    "mw_last_error": (C.c_char_p, []),
    "mw_launch_count": (C.c_uint64, []),
    "mw_logmel_plan_create": (C.c_int32, [C.c_int, c_f32p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "mw_logmel_plan_destroy": (None, [C.c_void_p]),
    "mw_logmel": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int,
                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "mw_logmel_long": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "mw_model_create": (C.c_int32, [C.POINTER(ModelConfigC), C.POINTER(WeightTableC), C.POINTER(C.c_void_p)]),
    "mw_model_destroy": (None, [C.c_void_p]),
    "mw_model_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "mw_encode": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_encode_t": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_generate": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, c_i32p, C.c_int, C.POINTER(GenOptionsC),
                                c_i32p, c_i32p, c_f32p, C.c_void_p]),
    "mw_decoder_logits": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, c_i32p, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_detect_language": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, C.c_int32, C.c_int32, C.c_int32,
                                       c_f32p, C.c_void_p]),
    "mw_gemm_h16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mw_decode_gemm_h16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_void_p]),
    "mw_decode_gemm_debug": (None, [C.c_void_p]),
    "mw_debug_step_parts": (None, [C.c_int]),
    "mw_set_solo": (C.c_int32, [C.c_void_p, C.c_int]),
    "mw_attention_h16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mw_bench_kernel": (C.c_int32, [C.c_void_p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_void_p]),
    "mw_bench_step": (C.c_int32, [C.c_void_p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_void_p]),
    "mw_frame_rms": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_vad_windows": (C.c_int32, [C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_double, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_layernorm": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "mw_gemm_general_h16": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                        C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_void_p]),
    "mw_attention_general_h16": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p,
                                             C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_layernorm_mode": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mw_step_projection_h16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "mw_step_self_attention_h16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_void_p]),
    "mw_step_prefill_attention_h16": (C.c_int32, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "mw_step_cross_attention_h16": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                C.c_void_p]),
    "mw_w2v_create": (C.c_int32, [C.POINTER(W2vConfigC), C.POINTER(WeightTableC), C.POINTER(C.c_void_p)]),
    "mw_w2v_destroy": (None, [C.c_void_p]),
    "mw_w2v_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "mw_w2v_frames": (C.c_int32, [C.c_int64]),
    "mw_w2v_emissions": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, c_i32p, C.c_int, C.c_void_p,
                                     C.c_int64, C.c_void_p]),
    "mw_w2v_debug_copy": (C.c_int32, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "mw_pcm_resample": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                    C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "mw_ctc_align": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
}


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Load libmw_b200.so, declaring every signature.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -m manual_whisper_b200.build` "
            "(nvcc, sm_100a). This package has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(_LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.mw_abi_version() != 2:
        raise RuntimeError(f"libmw_b200.so ABI version {lib.mw_abi_version()} != 2 (rebuild: python -m manual_whisper_b200.build)")
    _lib = lib
    return lib


def check(status: int, what: str):
    if status != 0:
        msg = load().mw_last_error().decode("utf-8", "replace")
        if status == 1:
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed (status {status}): {msg}")


def storage_dtype():
    """torch dtype of the engine's 16-bit buffers (include/mw_b200.h: mw_storage_dtype): float16 unless the library was
    built with MW_STORAGE_BF16=1."""
    import torch
    return torch.bfloat16 if load().mw_storage_dtype() == 1 else torch.float16


def launch_count() -> int:
    return int(load().mw_launch_count())
