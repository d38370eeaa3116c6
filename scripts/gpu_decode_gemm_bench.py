#!/usr/bin/env python3
"""Isolated timing of the weight-stationary decode GEMM (csrc/decode_gemm.cu) at large-v3 shapes.
CUDA events on the launching stream, weights cycled over enough copies to exceed the 126 MB L2.  JSON to stdout."""
import ctypes as C, json, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from manual_whisper_b200 import _lib
lib = _lib.load(); dev = torch.device("cuda:0"); H = _lib.storage_dtype()
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
shapes = {"dxd": (1280, 1280), "qkv": (3840, 1280), "fc1": (5120, 1280), "fc2": (1280, 5120), "logits": (51866, 1280)}
out = []
for name, (N, K) in shapes.items():
    copies = max(2, int(260e6 // (N * K * 2)) + 1)
    w = (torch.randn(copies, N, K, device=dev) * 0.02).to(H)
    bias = torch.randn(N, device=dev)
    for R in (32, 64, 128, 256):
        x = (torch.randn(R, K, device=dev) * 0.5).to(H)
        o = torch.empty(R, N, device=dev, dtype=H)
        def run(i):
            _lib.check(lib.mw_decode_gemm_h16(x.data_ptr(), w[i % copies].data_ptr(), bias.data_ptr(), None, o.data_ptr(), R, N, K, 0, st), "dg")
        for i in range(5): run(i)
        iters = 4 * copies if N < 10000 else 24
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters): run(i)
        e1.record(); torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / iters
        out.append({"gemm": name, "N": N, "K": K, "R": R, "us": round(us, 2), "weight_GBps": round(N * K * 2 / us / 1e3, 1),
                    "TFLOPs": round(2.0 * R * N * K / us / 1e6, 1)})
        print(out[-1], file=sys.stderr, flush=True)
print(json.dumps({"rows": out}))
