"""Decode-step anatomy with MERGED device batches: S replicas (shared weights, one stream + host thread each) of ROWS rows
replay one kernel class of the step concurrently.  Reports ms per step and ms per 32-window batch-step equivalent.
args: ROWS S [iters] [classes]"""
import sys, json, threading
import torch
sys.path.insert(0, ".")
import manual_whisper_b200 as mw
from manual_whisper_b200.config import model_dims
from bench import device_weights, MODEL
ROWS = int(sys.argv[1]); S = int(sys.argv[2])
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 20
only = sys.argv[4].split(",") if len(sys.argv) > 4 else None
dev = torch.device("cuda:0"); dims = model_dims(MODEL)
pipe = mw.load_model(MODEL, "cuda", compute_type="float16", language="zh", asr_options={"beam_size": 1},
                     vad_model=mw.InjectedVad([]), model=device_weights(dims, dev, seed=1234), max_batch=ROWS, streams_per_device=S)
res = {"rows": ROWS}
for parts, name in [(4, "gemm"), (16, "cross"), (2, "ln"), (8, "self"), (32, "logits"), (63, "layers+logits")]:
    if only and name not in only:
        continue
    for n in sorted({1, S}):
        out = [0.0] * n
        def work(i):
            rep = pipe.replicas[i]
            s = rep.stream or torch.cuda.current_stream(rep.device)
            with torch.cuda.device(rep.device), torch.cuda.stream(s):
                out[i] = rep.engine.bench_step(ROWS, parts, iters)
        th = [threading.Thread(target=work, args=(i,)) for i in range(n)]
        [t.start() for t in th]; [t.join() for t in th]
        ms = max(out)
        res[f"{name}_x{n}"] = {"ms_per_step_each": round(ms, 3), "ms_per_32row_batch_step": round(ms / n / (ROWS / 32.0), 3)}
print(json.dumps(res))
