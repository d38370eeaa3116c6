"""The C-ABI library builds, loads and exports every symbol include/mw_b200.h declares (no GPU needed)."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "mw_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mw_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_three_seams():
    syms = header_symbols()
    for s in ("mw_logmel", "mw_logmel_long", "mw_encode", "mw_generate", "mw_model_create", "mw_model_destroy",
              "mw_last_error", "mw_abi_version"):
        assert s in syms


def test_library_exports_every_declared_symbol(built_lib):
    out = subprocess.check_output(["nm", "-D", "--defined-only", str(built_lib)], text=True)
    exported = set(re.findall(r" T (mw_[a-z0-9_]+)", out))
    missing = [s for s in header_symbols() if s not in exported]
    assert not missing, f"declared in include/mw_b200.h but not exported: {missing}"


def test_ctypes_signatures_cover_header(built_lib):
    from manual_whisper_b200 import _lib
    assert sorted(_lib.SIGNATURES) == header_symbols()
    lib = _lib.load()
    assert lib.mw_abi_version() == 2
    assert lib.mw_storage_dtype() in (0, 1)
    assert isinstance(lib.mw_launch_count(), int)


def test_argument_errors_do_not_need_a_gpu(built_lib):
    from manual_whisper_b200 import _lib
    lib = _lib.load()
    handle = C.c_void_p()
    st = lib.mw_logmel_plan_create(128, None, 4, 0, C.byref(handle))
    assert st == 1 and b"null" in lib.mw_last_error()
    with pytest.raises(ValueError):
        _lib.check(st, "mw_logmel_plan_create")
    assert lib.mw_model_create(None, None, C.byref(handle)) == 1
    assert lib.mw_logmel(None, None, 0, None, None, 1, None, None, None) == 1


def test_step_entry_points_reject_bad_arguments_without_a_gpu(built_lib):
    """Shapes, paths and pointers are checked before anything touches the device; every call here is rejected up front."""
    from manual_whisper_b200 import _lib
    lib = _lib.load()
    proj = lib.mw_step_projection_h16
    # forced kernels that do not exist for K (checked before the pointers, which are null here)
    # (gamma and beta only mark the LayerNorm path: x, W and out are null, so nothing could be launched)
    for path, K in [(4, 640), (5, 1536), (5, 2048), (6, 1280), (7, 640), (7, 2560), (9, 1536), (9, 2048)]:
        g = 16 if path == 9 else None
        assert proj(None, None, g, g, None, None, None, None, 32, 64, K, 0, path, None) == 3, (path, K)
        assert b"no " in lib.mw_last_error() and str(K).encode() in lib.mw_last_error()
    assert proj(None, None, 16, 16, None, None, None, None, 32, 64, 512, 2, 9, None) == 3    # fused LN has no fp32 output
    # bad shapes, flags and paths
    assert proj(None, None, None, None, None, None, None, None, 32, 64, 100, 0, 0, None) == 1
    assert proj(None, None, None, None, None, None, None, None, 0, 64, 128, 0, 0, None) == 1
    assert proj(None, None, None, None, None, None, None, None, 32, 64, 128, 4, 0, None) == 1
    assert proj(None, None, None, None, None, None, None, None, 32, 64, 128, 0, 11, None) == 1
    assert proj(None, None, None, None, None, None, None, None, 32, 64, 128, 0, 10, None) == 1    # LN path without gamma
    # supported shapes with null pointers
    for path in range(9):
        K = 2048 if path in (6, 7) else 512
        assert proj(None, None, None, None, None, None, None, None, 32, 64, K, 0, path, None) == 1
        assert b"null" in lib.mw_last_error()
    assert lib.mw_step_self_attention_h16(None, None, None, None, 4, 6, 448, 0, None, None) == 1
    assert b"null" in lib.mw_last_error()
    assert lib.mw_step_self_attention_h16(None, None, None, None, 4, 6, 448, 448, None, None) == 1     # pos outside ctx
    assert lib.mw_step_prefill_attention_h16(None, 2, 16, 6, None, None) == 1
    cross = lib.mw_step_cross_attention_h16
    assert cross(None, None, 2, 9, 1500, 6, 4, None, None) == 1 and b"G=9" in lib.mw_last_error()
    assert cross(None, None, 2, 0, 1500, 6, 4, None, None) == 1
    assert cross(None, None, 2, 1, 1500, 6, 2, None, None) == 1 and b"unr" in lib.mw_last_error()
    assert cross(None, None, 2, 1, 1500, 6, 8, None, None) == 1 and b"null" in lib.mw_last_error()


def test_sass_is_blackwell_native(built_lib):
    """tcgen05.mma -> UTCHMMA, tcgen05.ld -> LDTM, TMA -> UTMALDG must be present in the sm_100a SASS."""
    sass = subprocess.check_output(["cuobjdump", "-sass", str(built_lib)], text=True)
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in sass, f"{mnemonic} missing: the GEMM/attention kernels are not on the tcgen05/TMA path"


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "manual_whisper_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"
