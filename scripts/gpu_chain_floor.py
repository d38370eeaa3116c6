"""Per-node cost of a serial chain of short kernels inside a CUDA graph (what bounds the single-stream decode step):
N dependent LayerNorm launches (rows x 1280) captured into one graph and replayed."""
import ctypes as C, json, os, sys
import torch
sys.path.insert(0, os.environ.get("GRAFT_REPO_ROOT", "/root/repo"))
from manual_whisper_b200 import _lib
lib = _lib.load(); dev = torch.device("cuda:0"); H = _lib.storage_dtype()
N = 1000
out = {}
for rows in (1, 8, 32, 160):
    x = torch.randn(rows, 1280, device=dev); g = torch.ones(1280, device=dev); b = torch.zeros(1280, device=dev)
    o = torch.empty(rows, 1280, device=dev, dtype=H)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        st = C.c_void_p(s.cuda_stream)
        for _ in range(3): _lib.check(lib.mw_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), o.data_ptr(), rows, 1280, st), "ln")
        s.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            st2 = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            for _ in range(N): _lib.check(lib.mw_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), o.data_ptr(), rows, 1280, st2), "ln")
        for _ in range(3): gr.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); 
        for _ in range(5): gr.replay()
        e1.record(); torch.cuda.synchronize()
        out[f"rows{rows}_us_per_node"] = round(e0.elapsed_time(e1) / 5 / N * 1e3, 3)
print(json.dumps(out))
