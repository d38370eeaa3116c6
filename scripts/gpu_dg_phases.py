"""Phase timestamps (%globaltimer, ns) of CTA (0,0) of the decode GEMM: where a ~10 us kernel spends its time."""
import ctypes as C, json, os, sys
import torch
sys.path.insert(0, os.environ.get("GRAFT_REPO_ROOT", "/root/repo"))
from manual_whisper_b200 import _lib
lib = _lib.load(); dev = torch.device("cuda:0"); H = _lib.storage_dtype()
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
stamps = torch.zeros(8, dtype=torch.int64, device=dev)
lib.mw_decode_gemm_debug(stamps.data_ptr())
names = ["setup", "loads+mma", "cluster_bar1", "scatter", "cluster_bar2", "reduce+store", "dealloc"]
for (N, K) in ((1280, 1280), (1280, 5120), (5120, 1280)):
    w = (torch.randn(4, N, K, device=dev) * 0.02).to(H); bias = torch.randn(N, device=dev)
    for R in (32, 128, 256):
        x = (torch.randn(R, K, device=dev) * 0.5).to(H); o = torch.empty(R, N, device=dev, dtype=H)
        acc = None
        for i in range(6):
            flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev).fill_(1)      # evict W from L2
            _lib.check(lib.mw_decode_gemm_h16(x.data_ptr(), w[i % 4].data_ptr(), bias.data_ptr(), None, o.data_ptr(), R, N, K, 0, st), "dg")
            torch.cuda.synchronize()
            t = stamps.cpu().numpy()
            d = [int(t[j + 1] - t[j]) for j in range(7)]
            if i >= 2:
                acc = d if acc is None else [a + b for a, b in zip(acc, d)]
        print(json.dumps({"N": N, "K": K, "R": R, "ns": {n: round(a / 4) for n, a in zip(names, acc)}, "total_ns": round(sum(acc) / 4)}))
lib.mw_decode_gemm_debug(None)
