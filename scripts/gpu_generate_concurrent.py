"""Decode phase alone, as the pipeline runs it: S shared-weight replicas each call engine.generate (224 greedy steps, 32 rows)
REP times from their own host thread + stream; optionally E extra threads run the encoder in a loop at the same time.
Prints aggregate ms per 32-window batch and per decode step.  args: S [REP] [E]   env ROWS = rows per replica (default 32),
PARTS = kernel classes kept in the step graphs (mask of mw_debug_step_parts, default 127 = the real step; ids are then meaningless)"""
import sys, json, threading, time
import torch
sys.path.insert(0, ".")
import manual_whisper_b200 as mw
from manual_whisper_b200.config import model_dims, special_tokens
from manual_whisper_b200 import _lib
from bench import device_weights, MODEL
import os
BATCH = int(os.environ.get("ROWS", "32")); PARTS = int(os.environ.get("PARTS", "127"))
S = int(sys.argv[1]); REP = int(sys.argv[2]) if len(sys.argv) > 2 else 3; E = int(sys.argv[3]) if len(sys.argv) > 3 else 0
dev = torch.device("cuda:0"); dims = model_dims(MODEL); tok = special_tokens(dims.vocab)
pipe = mw.load_model(MODEL, "cuda", compute_type="float16", language="zh", asr_options={"beam_size": 1},
                     vad_model=mw.InjectedVad([]), model=device_weights(dims, dev, seed=1234), max_batch=BATCH, streams_per_device=S + E)
_lib.load().mw_debug_step_parts(PARTS)
prompt = [tok.sot, tok.lang_id("zh"), tok.transcribe, tok.no_timestamps]
feat_t = torch.randn(BATCH, 3002, dims.n_mels, device=dev).to(pipe.model.engine.h16)
encs = []
for rep in pipe.replicas:
    with torch.cuda.stream(rep.stream):
        encs.append(rep.engine.encode_time_major(feat_t))
        rep.engine.generate(encs[-1], prompt, tok, beam_size=1)          # graph capture, warm-up
torch.cuda.synchronize()
stop = threading.Event(); enc_count = [0] * E
def gen(i):
    rep = pipe.replicas[i]
    with torch.cuda.device(dev), torch.cuda.stream(rep.stream):
        for _ in range(REP):
            rep.engine.generate(encs[i], prompt, tok, beam_size=1)
def enc(j):
    rep = pipe.replicas[S + j]
    with torch.cuda.device(dev), torch.cuda.stream(rep.stream):
        while not stop.is_set():
            rep.engine.encode_time_major(feat_t); rep.stream.synchronize(); enc_count[j] += 1
th = [threading.Thread(target=gen, args=(i,)) for i in range(S)]
te = [threading.Thread(target=enc, args=(j,)) for j in range(E)]
t0 = time.perf_counter()
[t.start() for t in te]; [t.start() for t in th]; [t.join() for t in th]
torch.cuda.synchronize(); dt = time.perf_counter() - t0
stop.set(); [t.join() for t in te]
n = S * REP
print(json.dumps({"streams": S, "encoder_threads": E, "batches": n, "rows": BATCH, "ms_per_32row_batch": round(dt / n * 1e3 / (BATCH / 32.0), 1),
                  "ms_per_32row_step": round(dt / n / 224 * 1e3 / (BATCH / 32.0), 3), "encodes_done": sum(enc_count),
                  "parts": PARTS}))
