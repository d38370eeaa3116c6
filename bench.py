#!/usr/bin/env python3
"""bench.py — RTFx of the hot path on N B200s (driver contract in the task statement).

Workload (BASELINE.json configs[2], "the configuration the metric is quoted on"): Whisper large-v3, a 1-hour
synthetic 16 kHz recording (speech-like bursts, SURVEY.md §8d C3), VAD turns injected from the generator and merged
into <=30 s windows, batch_size=32, greedy decoding, random-init weights (no checkpoint offline).

N = 1
  step   = one batch of 32 windows through log-mel -> encoder -> greedy decode (224 tokens: random-init weights never
           emit <eot>, so every window decodes to the cap - worst case).  --streams batches (default 8) are kept in
           flight (shared-weight replicas, one stream each); ms_per_step = timed region / K.
  value  = audio seconds of the windows processed in the K timed steps / device time, inputs resident in HBM.
  e2e    = the same metric through the public API model.transcribe(host_audio, batch_size=32): pinned host waveform
           -> H2D -> windows -> ids back on the host, for the whole hour.
N > 1 (torchrun, one process per GPU)
  value  = STRONG scaling, what BASELINE config 3 / the north star name: ONE 1-hour recording, its ~136 windows sharded
           over the ranks (longest-first bin packing, manual_whisper_b200/distributed.py), each rank's share resident in
           its HBM; a step = one pass of every rank over its share; device time, max over ranks.  The ids gathered on
           rank 0 are checked equal to a single-GPU pass ("ids_match_single_gpu").
  e2e    = distributed.transcribe_sharded(host_audio): H2D of each rank's span, decode, all_gather_object of the ids.
  weak   = the round-1 number beside it: every rank transcribes its OWN hour (trivially linear).
Extra objects on the line: roofline (dominant kernel, HBM), roofline.tensor (encoder), roofline.in_step (cost of
each kernel class inside the real concurrent decode loop), logmel (the metric's second half), cpu_baseline.

--impl reference times the reference's CPU configuration (/root/reference/transcribe.py:29-32: cpu / int8 /
batch_size 4) on the host cores with the oracle port (the reference's own stack, whisperx / faster-whisper /
CTranslate2, is not installable offline): a step = one batch of 4 windows, log-mel + encoder + cross-K/V + all 224
greedy tokens, dynamic int8 Linear layers, every core.  Everything it prints is measured; nothing is extrapolated.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = "large-v3"
BATCH = 32
CPU_BATCH = 4          # the reference's BATCH_SIZE default (/root/reference/transcribe.py:31)
HOUR_S = 3600.0
MAX_NEW = 224
METRIC = "RTFx (audio-s/wall-s) Whisper large-v3 batched"
WORKLOAD = (f"{MODEL} (128 mels), 1-hour synthetic 16 kHz recording, VAD-chunked into <=30 s windows, "
            f"batch_size={BATCH}, greedy, {MAX_NEW} tokens/window (random-init weights never emit eot)")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "tensor_burst": float(d["bf16_tflops"]),
                "tensor_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def _dist():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def device_weights(dims, dev, seed):
    """Random-init large-v3 weights generated on the device (SURVEY.md §8d: N(0, 0.02^2), LN gamma=1 beta=0), rounded once to
    the 16-bit grid the engine stores (manual_whisper_b200/weights.py: round_shared)."""
    from manual_whisper_b200.weights import _keys, sinusoids, round_shared
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    sd = {}
    for name, shape, kind in _keys(dims):
        if kind == "g":
            sd[name] = torch.ones(shape, device=dev)
        elif kind == "beta":
            sd[name] = torch.zeros(shape, device=dev)
        else:
            sd[name] = round_shared(torch.randn(shape, device=dev, generator=g) * 0.02)
    sd["model.encoder.embed_positions.weight"] = sinusoids(dims.n_audio_ctx, dims.d_model).to(dev)
    return sd


# ----------------------------------------------------------------------------------------------- CPU legs
class CpuReference:
    """The reference's CPU configuration restated with the oracle: one step = one batch of CPU_BATCH windows of the
    1-hour recording through log-mel -> encoder -> cross-K/V -> prefill -> all MAX_NEW greedy tokens."""

    def __init__(self, int8: bool = True):
        from manual_whisper_b200.config import model_dims, special_tokens
        from manual_whisper_b200.vad import synthetic_speech, merge_chunks
        from manual_whisper_b200.weights import _keys, sinusoids
        self.dims = dims = model_dims(MODEL)
        tok = special_tokens(dims.vocab)
        g = torch.Generator().manual_seed(1234)
        sd = {}
        for name, shape, kind in _keys(dims):
            if kind == "g":
                sd[name] = torch.ones(shape)
            elif kind == "beta":
                sd[name] = torch.zeros(shape)
            else:
                sd[name] = torch.empty(shape).normal_(0.0, 0.02, generator=g)
        sd["model.encoder.embed_positions.weight"] = sinusoids(dims.n_audio_ctx, dims.d_model)
        self.sd = sd
        self.models = {}
        self.model(int8)
        audio, turns = synthetic_speech(CPU_BATCH * 40.0 * 3, seed=1)
        wins = merge_chunks(turns, 30)
        self.windows = [audio[int(w["start"] * 16000): int(w["end"] * 16000)] for w in wins]
        self.prompt = [tok.sot, tok.lang_id("zh"), tok.transcribe, tok.no_timestamps]

    def model(self, int8):
        from oracle.model import OracleWhisper
        if int8 not in self.models:
            self.models[int8] = OracleWhisper(self.dims, self.sd, int8=int8)
        return self.models[int8]

    def step(self, index: int, int8: bool = True, threads: int = 0, decode_steps: int = MAX_NEW):
        """-> (audio seconds, wall seconds, parts)"""
        from oracle.logmel import log_mel_spectrogram
        torch.set_num_threads(threads or (os.cpu_count() or 1))
        orc = self.model(int8)
        ws = [self.windows[(index * CPU_BATCH + i) % len(self.windows)] for i in range(CPU_BATCH)]
        secs = sum(len(a) for a in ws) / 16000.0
        t0 = time.perf_counter()
        with torch.no_grad():
            mel = torch.stack([log_mel_spectrogram(a, self.dims.n_mels, padding=480000 - len(a)) for a in ws])
            t1 = time.perf_counter()
            enc = orc.encode(mel)
            t2 = time.perf_counter()
            cross = orc.cross_kv(enc)
            cache = orc.new_cache()
            orc.decode(torch.tensor([self.prompt[:-1]] * CPU_BATCH), 0, cross, cache)
            cur = torch.tensor([[self.prompt[-1]]] * CPU_BATCH)
            t3 = time.perf_counter()
            for s in range(decode_steps):
                lg = orc.decode(cur, len(self.prompt) - 1 + s, cross, cache)[:, 0]
                cur = lg.argmax(-1, keepdim=True)
            t4 = time.perf_counter()
        return secs, t4 - t0, {"logmel_s": t1 - t0, "encoder_s": t2 - t1, "cross_kv_prefill_s": t3 - t2,
                               "decode_s": t4 - t3, "decode_steps": decode_steps, "decode_s_per_token": (t4 - t3) / max(decode_steps, 1)}


def _cpu_desc(int8, threads, decode_steps=MAX_NEW):
    return (f"one batch of {CPU_BATCH} windows (the reference's BATCH_SIZE) of the recording: log-mel + large-v3 encoder + cross-K/V "
            f"+ prefill + {decode_steps} greedy tokens, all measured; "
            f"{'dynamic int8 Linear layers (the reference ships compute_type int8)' if int8 else 'fp32'}, "
            f"{threads} threads; torch CPU restatement (oracle/), not CTranslate2")


def run_reference(args):
    rank, world, _ = _dist()
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    ref = CpuReference(int8=True)
    ref.step(0, decode_steps=1)        # untimed: packs the int8 weights (done lazily, once per Linear) and pages everything in
    t, audio, parts = [], 0.0, None
    for i in range(args.steps):
        secs, dt, parts = ref.step(1 + i)
        audio += secs
        t.append(dt)
    total = sum(t)
    v = audio / total
    variants = {}
    # the driver's scaling run gives every arm 870 s: with K >= 10 full-length steps (~24 s each on 16 cores) the variant rows
    # (another ~40 s) are left to the default invocation
    if not args.no_variants and args.steps < 10:
        # the same batch once each with 32 tokens: the reference's default thread count (whisperx threads=4) and plain fp32
        for name, int8, threads in (("int8_all_cores", True, cores), ("int8_threads4", True, 4), ("fp32_all_cores", False, cores)):
            secs, dt, p = ref.step(0, int8=int8, threads=threads, decode_steps=32)
            variants[name] = {"seconds": dt, "audio_s": secs, "parts": p}
        variants["note"] = "bounded rows (32 decode tokens each): compare encoder_s and decode_s_per_token across rows"
    line = {"metric": METRIC, "impl": "reference", "value": v, "unit": "x real-time",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / len(t) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "weights": "random-init N(0,0.02^2) seed 1234", "sample": _cpu_desc(True, cores),
                       "reference_config": "DEVICE=cpu COMPUTE_TYPE=int8 BATCH_SIZE=4 (/root/reference/transcribe.py:29-32)"},
            "cpu_baseline": {"value": v, "unit": "x real-time", "cores": cores, "kind": "port", "sample": _cpu_desc(True, cores),
                             "parts_last_step": parts, "variants": variants},
            "e2e": {"value": v, "unit": "x real-time", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------- GPU extras (rank 0, N = 1)
def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def measure_logmel(model, dims, hbm, cpu: bool):
    """The metric's second half: log-mel GB/s of ALGORITHMIC bytes (4 N + 4 n_mels N/160), CUDA events on the launching stream."""
    from manual_whisper_b200 import audio as A
    dev = model.device
    n_w = BATCH
    g = torch.Generator(device=dev).manual_seed(5)
    clip = torch.randn(n_w * 480000, device=dev, generator=g) * 0.1
    offs = torch.arange(n_w, dtype=torch.int64, device=dev) * 480000
    lens = torch.full((n_w,), 480000, dtype=torch.int32, device=dev)
    feat = torch.empty(n_w, dims.n_mels, 3000, device=dev)
    feat_t = torch.empty(n_w, 3002, dims.n_mels, device=dev, dtype=model.engine.h16)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {}

    def timed(fn, iters=10):
        for _ in range(3):
            fn()
        ms = []
        for _ in range(iters):
            flush.fill_(1)                      # evict: the next call reads its audio from HBM
            e0, e1 = _events()
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return statistics.median(ms)

    ms = timed(lambda: model.plan.chunks(clip, offs, lens, out=feat, out_t=feat_t))
    nbytes = n_w * (4 * 480000 + 4 * dims.n_mels * 3000)
    out["chunked_32x30s"] = {"ms": ms, "GBps": nbytes / ms / 1e6, "frac_of_hbm": nbytes / ms / 1e6 / hbm, "bytes": nbytes,
                             "what": "mw_logmel: 32 windows of 30 s, per-window max, f32 + 16-bit time-major outputs; L2 flushed between calls"}
    hour = torch.randn(int(HOUR_S) * 16000, device=dev, generator=g) * 0.1
    plan = A.get_plan(dims.n_mels, dev)
    ms = timed(lambda: plan.long(hour, padding=0), iters=5)
    nbytes = 4 * hour.numel() + 4 * dims.n_mels * (hour.numel() // 160)
    out["unchunked_1h"] = {"ms": ms, "GBps": nbytes / ms / 1e6, "frac_of_hbm": nbytes / ms / 1e6 / hbm, "bytes": nbytes,
                           "what": "mw_logmel_long: log_mel_spectrogram(audio[1 h], padding=0), one global max (config 5); values are stored "
                                   "scaled and only tiles holding a value below max - 8 are revisited (noise-like audio: a handful)"}
    hour.view(-1, 160000)[:, 80000:] = 0.0          # 5 s of digital silence in every 10 s: the clamp has work to do
    ms = timed(lambda: plan.long(hour, padding=0), iters=5)
    out["unchunked_1h_with_silence"] = {"ms": ms, "GBps": nbytes / ms / 1e6, "frac_of_hbm": nbytes / ms / 1e6 / hbm, "bytes": nbytes,
                                        "what": "the same call on a clip that is half digital silence: every tile with silence is "
                                                "clamped in a second in-place pass"}
    if cpu:
        from oracle.logmel import log_mel_spectrogram          # the torch.stft path of whisperx.audio.log_mel_spectrogram
        torch.set_num_threads(os.cpu_count() or 1)
        a = clip[: 8 * 480000].cpu().numpy()
        log_mel_spectrogram(a[:480000], dims.n_mels)
        t0 = time.perf_counter()
        for i in range(8):
            log_mel_spectrogram(a[i * 480000: (i + 1) * 480000], dims.n_mels)
        dt = time.perf_counter() - t0
        nb = 8 * (4 * 480000 + 4 * dims.n_mels * 3000)
        out["cpu_torch_stft"] = {"GBps": nb / dt / 1e9, "cores": os.cpu_count() or 1, "sample": "8 windows of 30 s, oracle/logmel.py (torch.stft)"}
    return out


def measure_encoder(model, dims, peaks):
    """roofline.tensor: the encoder (conv stem + 32 layers, tcgen05 GEMMs + attention) on one batch of 32 windows."""
    dev = model.device
    feat_t = (torch.randn(BATCH, 3002, dims.n_mels, device=dev) * 0.3).to(model.engine.h16)
    for _ in range(2):
        model.engine.encode_time_major(feat_t)
    ms = []
    for _ in range(5):
        e0, e1 = _events()
        e0.record(); model.engine.encode_time_major(feat_t); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = statistics.median(ms)
    d, T, L, F = dims.d_model, dims.n_audio_ctx, dims.enc_layers, dims.ffn
    flop = 2 * 3000 * d * 3 * dims.n_mels + 2 * T * d * 3 * d + L * (8 * T * d * d + 4 * T * T * d + 4 * T * d * F)   # SURVEY.md Appendix C
    tf = BATCH * flop / t / 1e9
    return {"bound": "tensor", "what": "mw_encode_t on 32 windows (activations of 123-492 MB per layer: larger than L2 between kernels)",
            "ms": t, "achieved": tf, "peak": peaks["tensor_sustained"], "unit": "TFLOP/s", "frac": tf / peaks["tensor_sustained"],
            "peak_kind": "sustained (a ~0.1 s kernel sequence inside a long step)", "flop_per_window": flop}


def measure_in_step(pipe, dims, tok, hbm, streams):
    """Cost of each kernel class INSIDE the real decode loop: `streams` replicas run mw_generate concurrently (as the timed
    region does) with all classes, then with one class removed from the step graphs (mw_debug_step_parts); the difference is
    what the class costs under real concurrency - unlike a kernel timed alone, it includes the contention."""
    from manual_whisper_b200 import _lib
    lib = _lib.load()
    prompt = [tok.sot, tok.lang_id("zh"), tok.transcribe, tok.no_timestamps]
    reps = pipe.replicas[:streams]
    dev = reps[0].device
    feat_t = (torch.randn(BATCH, 3002, dims.n_mels, device=dev) * 0.3).to(reps[0].engine.h16)
    encs = []
    for rep in reps:
        with torch.cuda.stream(rep.stream):
            encs.append(rep.engine.encode_time_major(feat_t))
    torch.cuda.synchronize()

    def run(parts):
        lib.mw_debug_step_parts(parts)

        def work(i):
            with torch.cuda.device(dev), torch.cuda.stream(reps[i].stream):
                reps[i].engine.generate(encs[i], prompt, tok, beam_size=1)
        dt = 0.0
        for _ in range(2):                                    # first round re-captures the graphs, the second is timed
            th = [threading.Thread(target=work, args=(i,)) for i in range(len(reps))]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            [t.start() for t in th]
            [t.join() for t in th]
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        return dt / len(reps) / MAX_NEW * 1e3                 # ms per 32-window batch-step, aggregate

    try:
        full = run(127)
        no_cross = run(127 & ~16)
        no_gemm = run(127 & ~4)
    finally:
        lib.mw_debug_step_parts(127)
    d, T = dims.d_model, dims.n_audio_ctx
    cross_bytes = BATCH * T * 2 * d * 2 * dims.dec_layers
    w_bytes = 2 * dims.dec_layers * (8 * d * d + 2 * d * dims.ffn)
    step_bytes = cross_bytes + w_bytes + 2 * dims.vocab * d + BATCH * dims.dec_layers * 2 * (MAX_NEW // 2) * d * 2
    c_ms, g_ms = max(full - no_cross, 1e-6), max(full - no_gemm, 1e-6)
    return {"how": f"{len(reps)} replicas x mw_generate concurrently (cross-K/V projection, prefill and 224 steps); step graphs re-captured "
                   "with one kernel class removed (mw_debug_step_parts); wall clock around the threads",
            "ms_per_batch_step": full, "ms_without_cross_attention": no_cross, "ms_without_projection_gemms": no_gemm,
            "cross_attention": {"ms": c_ms, "GBps": cross_bytes / c_ms / 1e6, "frac_of_hbm": cross_bytes / c_ms / 1e6 / hbm},
            "projection_gemms": {"ms": g_ms, "GBps": w_bytes / g_ms / 1e6, "frac_of_hbm": w_bytes / g_ms / 1e6 / hbm},
            "whole_step": {"bytes": step_bytes, "GBps": step_bytes / full / 1e6, "frac_of_hbm": step_bytes / full / 1e6 / hbm,
                           "what": "weights + cross-K/V + tied-embedding logits + self-K/V at the mean position, per 32-window batch-step"}}


def _traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, read from the tracked ncu summary."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        e = d.get(kernel)
        if e:
            return e["dram_bytes_per_launch"], e["source"]
    return None, None


def dump_outputs(out_dir, ids):
    """Writes the token ids of the windows of the last timed step to out_dir/token_ids.npy: one row per window, padded with
    -1, float32 (ids below 2^24 are exact).  They are what a caller of the timed path receives, so two builds run with the
    same arguments can be compared output for output."""
    rows = np.full((len(ids), max((len(t) for t in ids), default=0)), -1, dtype=np.float32)
    for i, t in enumerate(ids):
        rows[i, :len(t)] = t
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "token_ids.npy"), rows)


# ----------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="reference arm: skip the threads=4 / fp32 variant rows")
    ap.add_argument("--no-extras", action="store_true", help="skip the logmel / encoder / in-step measurements (profiling runs)")
    ap.add_argument("--e2e-repeats", type=int, default=1)
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: do not time the public-API pass")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the token ids of the last step's windows to DIR/token_ids.npy")
    ap.add_argument("--merge", type=int, default=1, help="user batches of 32 windows merged into one device batch (rows are independent)")
    ap.add_argument("--streams", type=int, default=0, help="batches in flight per GPU (shared-weight replicas); default 8 (4 for --config reference)")
    ap.add_argument("--config", default="north_star", choices=["north_star", "reference"],
                    help="north_star: greedy, 4-token prompt (BASELINE configs).  reference: the call shape of /root/reference/transcribe.py:"
                         "107-113 - whisperx defaults (beam_size 5, patience 1, without_timestamps) plus a ~60-token initial_prompt")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    ref_shape = args.config == "reference"
    if not args.streams:
        args.streams = 4 if ref_shape else 8          # beam 5 holds 160 rows of self-K/V per replica (21 GB of workspace each)
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    rank, world, local = _dist()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import manual_whisper_b200 as mw
    from manual_whisper_b200 import _lib
    from manual_whisper_b200.config import model_dims, special_tokens
    from manual_whisper_b200.distributed import shard_windows, transcribe_sharded, gather_ordered

    dims = model_dims(MODEL)
    tok = special_tokens(dims.vocab)
    sd = device_weights(dims, dev, seed=1234)
    storage = "bf16" if _lib.load().mw_storage_dtype() == 1 else "fp16"

    def pinned_audio(seed):
        audio_np, tr = mw.synthetic_speech(HOUR_S, seed=seed)
        pinned = torch.empty(len(audio_np), dtype=torch.float32, pin_memory=True)
        pinned.numpy()[:] = audio_np
        return pinned.numpy(), tr

    # the shared recording: strong scaling at N > 1, everything at N = 1
    audio_host, turns = pinned_audio(1)
    asr_options = {"beam_size": 1}
    if ref_shape:
        # no tokenizer.json offline: the prompt text is encoded one id per byte, so 60 ASCII characters = 60 prompt tokens,
        # about what the reference's Chinese domain-term prompt (transcribe.py:40) tokenises to
        import warnings
        warnings.filterwarnings("ignore", message="no tokenizer.json")
        asr_options = {"beam_size": 5, "patience": 1, "length_penalty": 1, "without_timestamps": True,
                       "initial_prompt": "meeting notes: quarterly revenue, churn, roadmap, hiring plan."[:60]}
    pipe = mw.load_model(MODEL, "cuda", device_index=local, compute_type="float16", language="zh",
                         asr_options=asr_options, vad_model=mw.InjectedVad(turns), model=sd, max_batch=BATCH * args.merge,
                         streams_per_device=args.streams)
    del sd
    model = pipe.model
    windows = mw.merge_chunks(turns, 30)
    offs = np.array([int(w["start"] * 16000) for w in windows], dtype=np.int64)
    lens = np.array([int(w["end"] * 16000) for w in windows], dtype=np.int64) - offs
    lens32 = lens.astype(np.int32)

    def barrier():
        torch.cuda.synchronize()
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def warm_replicas(resident, o, l):
        # every replica (stream) must have captured its decode graphs before a timed region: one untimed batch each
        for rep in pipe.replicas:
            with torch.cuda.device(rep.device):
                sl = slice(0, min(len(o), BATCH * args.merge))
                rep.transcribe_windows(resident["audio"][rep.device], torch.from_numpy(o[sl] - resident["lo"]).to(rep.device),
                                       torch.from_numpy(l[sl]).to(rep.device), pipe.tokenizer, pipe.options)
        torch.cuda.synchronize()

    def timed(fn):
        """fn() with a barrier + synchronize on both sides, CUDA events; -> (ms, fn's value, launches, clocks)"""
        sampler = ClockSampler(local)
        barrier()
        sampler.start()
        l0 = _lib.launch_count()
        e0, e1 = _events()
        e0.record()
        val = fn()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), val, _lib.launch_count() - l0, sampler.stop()

    def allreduce(vals, op):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if use_dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return t.tolist()

    def throughput_steps(resident, o, l32, l64, steps):
        """`steps` batches of 32 windows (cycling the full batches of a recording) through the in-flight replicas
        -> (ms, audio seconds, launches, clocks, (text, ids) of the last step's windows)"""
        n_full = len(o) // BATCH

        def run(first, count):
            idx = np.concatenate([np.arange(((first + i) % n_full) * BATCH, ((first + i) % n_full + 1) * BATCH) for i in range(count)])
            res = pipe.run_device_batches(resident, o[idx], l32[idx], BATCH * args.merge)
            return float(l64[idx].sum()) / 16000.0, res
        run(0, args.warmup)
        ms, (audio_s, res), launches, clocks = timed(lambda: run(args.warmup, steps))
        return ms, audio_s, launches, clocks, res[-BATCH:]

    line = {"metric": METRIC, "unit": "x real-time", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "vs_baseline": None, "dtype": storage, "data": "synthetic"}
    workload = WORKLOAD if not ref_shape else WORKLOAD.replace("greedy", "beam_size 5 / patience 1 / 61-token initial prompt (the reference's call shape)")
    config = {"workload": workload, "windows": len(windows), "mean_window_s": float(lens.mean()) / 16000,
              "weights": f"random-init N(0,0.02^2) seed 1234, {storage} storage, fp32 accumulation",
              "l2": "inputs larger than L2 (weights 3.1 GB + cross-K/V 7.9 GB streamed per step)"}

    if not use_dist:
        # ------------------------------------------------------------------ N = 1
        resident = pipe.upload(audio_host, offs, lens)        # untimed: `value` is measured with inputs resident in HBM
        warm_replicas(resident, offs, lens32)
        ms, audio_s, launches, clocks, last_step = throughput_steps(resident, offs, lens32, lens, args.steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, [toks for _, toks in last_step])
        # the whole recording once, resident (the N = 1 point of the strong-scaling curve)
        pipe.run_device_batches(resident, offs, lens32, BATCH)
        ms_hour, _, _, _ = timed(lambda: pipe.run_device_batches(resident, offs, lens32, BATCH))
        t_e2e, result = [], {"segments": []}
        for _ in range(0 if args.skip_e2e else max(1, args.e2e_repeats)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            result = pipe.transcribe(audio_host, batch_size=BATCH * args.merge, language="zh")
            torch.cuda.synchronize()
            t_e2e.append(time.perf_counter() - t0)
        e2e_s = min(t_e2e) if t_e2e else float("inf")
        n_batches = (len(windows) + BATCH - 1) // BATCH
        span = int(offs[-1] + lens[-1] - offs[0])
        d2h = sum(len(s["tokens"]) for s in result["segments"]) * 4
        config["parallelism"] = f"dp1 (one process per GPU, {args.streams} batches in flight per GPU)"
        line.update({"value": audio_s / (ms / 1e3), "ms_per_step": ms / args.steps, "scaling": "weak", "config": config,
                     "clocks": clocks, "gpu_launches": int(launches),
                     "one_recording": {"value": HOUR_S / (ms_hour / 1e3), "unit": "x real-time", "ms": ms_hour,
                                       "what": "the whole 1-hour recording once (136 windows in 5 batches), inputs resident: the N = 1 "
                                               "point of the strong-scaling curve that bench.py --gpus N reports"},
                     "e2e": {"value": HOUR_S / e2e_s, "unit": "x real-time", "h2d_bytes_per_step": int(span * 4 / n_batches),
                             "d2h_bytes_per_step": int(d2h / n_batches), "seconds_per_hour_of_audio": e2e_s,
                             "api": "manual_whisper_b200.load_model(...).transcribe(host_audio, batch_size=32)"}})
        peaks = _peaks()
        eng = model.engine
        d, T = dims.d_model, dims.n_audio_ctx
        cand = [("cross_attn_stream_kernel", 0, BATCH * T * 2 * d * 2, dims.dec_layers * MAX_NEW),
                ("skinny_gemm_kernel(fc1)", 1, dims.ffn * d * 2, 2 * dims.dec_layers * MAX_NEW),      # fc1 + fc2 (same bytes)
                ("skinny_gemm_kernel(d x d)", 2, d * d * 2, 6 * dims.dec_layers * MAX_NEW)]           # q|k|v counted as three
        kern = []
        for name, which, nbytes, per_step in cand:
            kms = eng.bench_kernel(which, BATCH, iters=96)
            kern.append({"kernel": name, "avg_ms": kms, "bytes_per_launch": nbytes, "GBps": nbytes / kms / 1e6,
                         "launches_per_step": per_step, "isolated_ms_per_step": kms * per_step})
        dom = kern[0]
        traffic, traffic_src = _traffic(dom["kernel"])
        roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["GBps"], "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": dom["GBps"] / peaks["hbm"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"],
                    "timing": "isolated launches cycling over the 32 layers' K/V (7.9 GB > L2), CUDA events on the launching stream; "
                              "in_step below is the same kernel's cost inside the real concurrent step",
                    "all": kern}
        if not args.no_extras and not ref_shape:
            roofline["tensor"] = measure_encoder(model, dims, peaks)
            roofline["in_step"] = measure_in_step(pipe, dims, tok, peaks["hbm"], args.streams)
            line["logmel"] = measure_logmel(model, dims, peaks["hbm"], cpu=not args.no_cpu_baseline)
        if ref_shape:
            args.no_cpu_baseline = True          # the CPU leg is the greedy configuration; not comparable to this call shape
        line["roofline"] = roofline
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            ref = CpuReference(int8=True)
            ref.step(0, decode_steps=1)        # untimed: packs the int8 weights (lazy, once per Linear)
            secs, dt, parts = ref.step(1)
            line["cpu_baseline"] = {"value": secs / dt, "unit": "x real-time", "cores": cores, "kind": "port",
                                    "sample": _cpu_desc(True, cores), "parts": parts}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------------- N > 1: strong scaling of ONE recording
    mine = np.array(shard_windows(lens, world)[rank], dtype=np.int64)
    o_m, l_m, l32_m = offs[mine], lens[mine], lens32[mine]
    resident = pipe.upload(audio_host, o_m, l_m)
    warm_replicas(resident, o_m, l32_m)
    pipe.run_device_batches(resident, o_m, l32_m, BATCH)

    def passes():
        out = None
        for _ in range(args.steps):
            out = pipe.run_device_batches(resident, o_m, l32_m, BATCH)
        return out
    ms, res_mine, launches, clocks = timed(passes)
    ms_max = allreduce([ms], "max")[0]
    launches_all = allreduce([float(launches)], "sum")[0]
    # ids gathered on the host in window order (the path's only exchange), checked against a single-GPU pass on rank 0
    ids = gather_ordered([(int(i), r[1]) for i, r in zip(mine, res_mine)], len(windows))
    match = None
    if rank == 0:
        full = pipe.upload(audio_host, offs, lens)
        single = pipe.run_device_batches(full, offs, lens32, BATCH)
        match = [r[1] for r in single] == ids
        del full
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ids)          # a step here is one pass over the whole recording
    t_e2e = []
    for _ in range(0 if args.skip_e2e else max(1, args.e2e_repeats)):
        barrier()
        t0 = time.perf_counter()
        transcribe_sharded(pipe, audio_host, BATCH, rank, world, language="zh")
        torch.cuda.synchronize()
        t_e2e.append(time.perf_counter() - t0)
    e2e_s = allreduce([min(t_e2e) if t_e2e else float("inf")], "max")[0]
    span = int((o_m + l_m).max() - o_m.min()) if len(mine) else 0
    h2d = allreduce([float(span * 4)], "sum")[0]
    # the weak number beside it: every rank its own hour
    own_audio, own_turns = pinned_audio(1 + rank) if rank else (audio_host, turns)
    own_w = mw.merge_chunks(own_turns, 30)
    oo = np.array([int(w["start"] * 16000) for w in own_w], dtype=np.int64)
    ol = np.array([int(w["end"] * 16000) for w in own_w], dtype=np.int64) - oo
    own_res = pipe.upload(own_audio, oo, ol)
    ms_w, audio_w, _, _, _ = throughput_steps(own_res, oo, ol.astype(np.int32), ol, args.steps)
    ms_w_max = allreduce([ms_w], "max")[0]
    audio_w_sum = allreduce([audio_w], "sum")[0]
    # config 5 at N GPUs: independent replicas, every rank the un-chunked log-mel of its own 1-hour clip (no exchange needed)
    lm = None
    if not args.no_extras:
        from manual_whisper_b200 import audio as A
        g = torch.Generator(device=model.device).manual_seed(5 + rank)
        hour = torch.randn(int(HOUR_S) * 16000, device=model.device, generator=g) * 0.1
        plan = A.get_plan(dims.n_mels, model.device)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=model.device)
        for _ in range(3):
            plan.long(hour, padding=0)
        t = []
        for _ in range(5):
            flush.fill_(1)
            e0, e1 = _events()
            e0.record(); plan.long(hour, padding=0); e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        peaks = _peaks()
        lm_ms = allreduce([statistics.median(t)], "max")[0]
        nb = world * (4 * hour.numel() + 4 * dims.n_mels * (hour.numel() // 160))
        lm = {"unchunked_1h_per_gpu": {"ms": lm_ms, "GBps": nb / lm_ms / 1e6, "frac_of_hbm": nb / lm_ms / 1e6 / (world * peaks["hbm"]),
                                       "bytes": nb, "what": f"config 5 at {world} GPUs: independent replicas, each rank log_mel_spectrogram("
                                                            "audio[1 h], padding=0) of its own clip; total algorithmic bytes / max time over ranks"}}
        del hour, flush
    if rank == 0:
        per_rank = [len(s) for s in shard_windows(lens, world)]
        config["parallelism"] = (f"dp{world}: ONE recording, {len(windows)} windows sharded {min(per_rank)}-{max(per_rank)} per GPU "
                                 f"(longest-first bin packing), {args.streams} replicas per GPU, host gather of the ids; no data-path collective")
        line.update({"value": args.steps * HOUR_S / (ms_max / 1e3), "ms_per_step": ms_max / args.steps, "scaling": "strong",
                     "config": config, "clocks": clocks, "gpu_launches": int(launches_all),
                     "ids_match_single_gpu": bool(match),
                     "limiting_factor": "each GPU holds under-filled batches (windows per GPU <= a few batches of 32): the 224 decode steps "
                                        "are a serial chain of graph nodes at >= 3.3 us each (~260 nodes, ~3.3 ms per step however few rows, "
                                        "with LayerNorm folded into the projections when a GPU holds a single batch: mw_set_solo), so the "
                                        "time of a pass stops falling once a GPU holds a single batch; no collective is involved",
                     "e2e": {"value": HOUR_S / e2e_s, "unit": "x real-time", "h2d_bytes_per_step": int(h2d),
                             "d2h_bytes_per_step": len(windows) * MAX_NEW * 4, "seconds_per_hour_of_audio": e2e_s,
                             "api": "manual_whisper_b200.distributed.transcribe_sharded(pipe, host_audio, 32, rank, world)"},
                     "weak": {"value": audio_w_sum / (ms_w_max / 1e3), "unit": "x real-time", "ms_per_step": ms_w_max / args.steps,
                              "what": "every rank transcribes its OWN 1-hour recording (batches of 32, 8 in flight): total audio / max time"}})
        if lm:
            line["logmel"] = lm
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()
    return 0


def _json_only_stdout():
    """Libraries (NCCL's version banner, warnings) write to fd 1; the driver wants exactly one JSON line there.
    Everything but our final print goes to stderr."""
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    return real


if __name__ == "__main__":
    _real_stdout = _json_only_stdout()
    _print = print

    def print(*a, **k):      # noqa: A001 - the one JSON line goes to the real stdout
        _print(*a, **{**k, "file": _real_stdout, "flush": True})

    sys.exit(main())
