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


def test_building_block_entry_points_reject_bad_arguments_without_a_gpu(built_lib):
    """mw_gemm_general_h16, mw_attention_general_h16 and mw_layernorm_mode check shapes, strides, column ranges and the mode
    before any pointer: every call here has null pointers and is rejected up front."""
    from manual_whisper_b200 import _lib
    lib = _lib.load()

    def gemm(ars=240, abs_=0, wrs=240, resid=None, rbr=0, ldr=0, obr=0, off=0, ldo=384, batch=1, M=3000, N=384, K=240):
        return lib.mw_gemm_general_h16(None, ars, abs_, None, wrs, None, resid, rbr, ldr, None, obr, off, ldo, batch, M, N, K,
                                       1, 0, None)

    assert gemm() == 1 and b"null" in lib.mw_last_error()                           # a good conv1 geometry, null pointers
    assert gemm(ars=80, abs_=3002 * 80, obr=3002, off=1, batch=3) == 1 and b"null" in lib.mw_last_error()
    for bad in (dict(N=48), dict(K=236), dict(M=0), dict(batch=0), dict(ars=84), dict(ars=0), dict(abs_=-8), dict(wrs=232),
                dict(ldo=376), dict(ldo=388), dict(off=-1), dict(batch=2, obr=3000, off=1), dict(resid=16, ldr=380),
                dict(resid=16, ldr=386), dict(resid=16, ldr=384, rbr=-1)):
        assert gemm(**bad) == 1, bad
        assert b"null" not in lib.mw_last_error(), bad

    def att(ldq=3 * 384, cq=0, ldkv=3 * 384, ck=384, cv=768, out_ld=384, B=2, Tq=1500, Tk=1500, H=6, lens=None):
        return lib.mw_attention_general_h16(None, ldq, cq, None, ldkv, ck, cv, None, out_ld, B, Tq, Tk, H, lens, None)

    assert att() == 1 and b"null" in lib.mw_last_error()
    assert att(ldq=384, ldkv=768, ck=0, cv=384, Tq=223) == 1 and b"null" in lib.mw_last_error()
    for bad in (dict(B=0), dict(Tq=0), dict(Tk=0), dict(H=0), dict(H=7), dict(cq=64 * 13), dict(cq=-64), dict(ck=-8),
                dict(cv=768 + 64), dict(ldq=384 + 4), dict(cq=4), dict(out_ld=320), dict(out_ld=388),
                dict(ldq=384, ldkv=768, ck=0, cv=384, Tq=223, lens=16)):
        assert att(**bad) == 1, bad
        assert b"null" not in lib.mw_last_error(), bad
    assert att(H=7) == 1 and b"do not fit" in lib.mw_last_error()
    assert att(Tq=223, lens=16) == 1 and b"Tq == Tk" in lib.mw_last_error()

    ln = lib.mw_layernorm_mode
    for mode, d in ((0, 2048), (1, 512), (2, 128), (3, 2048)):
        assert ln(None, None, None, None, 7, d, mode, None) == 1 and b"null" in lib.mw_last_error()
    for mode, d in ((1, 640), (2, 1024), (3, 2176), (0, 100), (3, 0), (4, 512), (-1, 512)):
        assert ln(None, None, None, None, 7, d, mode, None) == 1, (mode, d)
        assert b"null" not in lib.mw_last_error(), (mode, d)
    assert ln(None, None, None, None, -1, 512, 3, None) == 1 and b"null" not in lib.mw_last_error()


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


def test_library_reads_only_its_debug_switches_from_the_environment():
    """The decode step has one routing, chosen from the shapes and mw_set_solo; it launches every kernel the ordinary way."""
    csrc = os.path.join(ROOT, "manual_whisper_b200", "csrc")
    names, dependent_launch = set(), []
    for dirpath, _, files in os.walk(csrc):
        for f in files:
            src = open(os.path.join(dirpath, f)).read()
            names |= set(re.findall(r"getenv\(\s*\"(MW_\w+)\"", src))
            if "griddepcontrol" in src:
                dependent_launch.append(f)
    assert names == {"MW_STEPWISE_PREFILL", "MW_RESAMPLE_DIRECT", "MW_W2V_STOP"}
    assert not dependent_launch
