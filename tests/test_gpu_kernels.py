"""Each tensor-core kernel pinned on its own (through the C ABI).  The tcgen05 GEMM, the flash attention and LayerNorm are held
to the per-element float64 bounds of tests/test_gpu_tensor_core_paths.py, whose checks these tests run at their shapes; the
decode GEMM against a plain PyTorch fp32 reference."""
import ctypes as C

import pytest
import torch

from test_gpu_tensor_core_paths import MODES, check_gemm_contiguous, check_layernorm, check_self_attention

pytestmark = pytest.mark.gpu


def _h16():
    from manual_whisper_b200 import _lib
    return _lib.storage_dtype()


@pytest.fixture(scope="module")
def lib():
    from manual_whisper_b200 import _lib
    return _lib.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (1, 128, 64), (257, 384, 240), (1500, 1280, 1280), (3000, 1152, 384),
                                   (4096, 5120, 1280), (777, 256, 5120), (300, 64, 1024), (100, 32, 128)])
@pytest.mark.parametrize("mode", ["plain", "bias_gelu", "bias_resid_f32"])
def test_gemm(lib, M, N, K, mode):
    """The tcgen05 GEMM on contiguous operands against float64, element by element."""
    check_gemm_contiguous(lib, M, N, K, mode)


@pytest.mark.parametrize("R,N,K", [(32, 1280, 1280), (17, 384, 384), (64, 3840, 1280), (68, 1280, 5120), (128, 5120, 1280),
                                   (128, 1280, 1280), (136, 1280, 1280), (256, 1280, 5120), (200, 51866, 1280), (1, 128, 128),
                                   (96, 51865, 384), (33, 2048, 128), (128, 300, 192)])
@pytest.mark.parametrize("mode", ["plain_f32", "bias_gelu", "bias_resid_f32"])
def test_decode_gemm(lib, R, N, K, mode):
    """The weight-stationary decode GEMM (swap-AB tcgen05, cluster split-K) against torch fp32; deterministic across runs."""
    from manual_whisper_b200 import _lib
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(R * 7 + N)
    x = (torch.randn(R, K, device=dev, generator=g) * 0.5).to(_h16())
    w = (torch.randn(N, K, device=dev, generator=g) * 0.05).to(_h16())
    bias = torch.randn(N, device=dev, generator=g) if mode != "plain_f32" else None
    res = torch.randn(R, N, device=dev, generator=g) if mode == "bias_resid_f32" else None
    f32 = mode != "bias_gelu"
    flags = (1 if mode == "bias_gelu" else 0) | (2 if f32 else 0)
    outs = []
    for _ in range(2):
        out = torch.full((R, N), 7.0, device=dev, dtype=torch.float32 if f32 else _h16())
        _lib.check(lib.mw_decode_gemm_h16(x.data_ptr(), w.data_ptr(), bias.data_ptr() if bias is not None else None,
                                          res.data_ptr() if res is not None else None, out.data_ptr(), R, N, K, flags, _stream()),
                   "mw_decode_gemm_h16")
        torch.cuda.synchronize()
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    ref = x.float() @ w.float().t()
    if bias is not None:
        ref = ref + bias
    if mode == "bias_gelu":
        ref = torch.nn.functional.gelu(ref)
    if res is not None:
        ref = ref + res
    tol = 2e-4 * ref.abs().max().item() if f32 else 2 ** -8 * ref.abs().max().item() + 1e-3
    assert (outs[0].float() - ref).abs().max().item() <= tol


def test_gemm_rejects_bad_shapes(lib):
    from manual_whisper_b200 import _lib
    t = torch.zeros(64, 64, device="cuda", dtype=_h16())
    assert lib.mw_gemm_h16(t.data_ptr(), t.data_ptr(), None, None, t.data_ptr(), 64, 48, 64, 0, 0, _stream()) == 1
    assert b"multiple of 32" in lib.mw_last_error()


@pytest.mark.parametrize("B,T,H", [(1, 128, 1), (1, 200, 2), (3, 1500, 6), (1, 1500, 20), (2, 77, 4)])
def test_encoder_attention(lib, B, T, H):
    """The flash attention on packed qkv against float64 with random scores and with every score pattern of
    tests/test_gpu_tensor_core_paths.py (lazy rescale at every key block, peaks at the first / last key, low, huge and
    fp16-subnormal probabilities)."""
    for mode in MODES:
        check_self_attention(lib, B, T, H, mode)


@pytest.mark.parametrize("rows,d", [(1, 128), (1000, 384), (37, 1280), (48000, 1280),
                                    (33, 512), (33, 640), (33, 1536), (33, 2048)])    # the MAXV boundaries of layernorm_launch
def test_layernorm(lib, rows, d):
    check_layernorm(lib, rows, d)
