"""Encoder / decoder / search parity of the CUDA engine against the oracle on the same bf16-rounded weights.

Stated tolerances (BASELINE.json north_star: "encoder output within stated bf16 tolerance", "greedy ids identical
on >= 99 % of chunks with divergences logged"):
  * encoder output: relative L2 error <= 2e-2 against the fp32 oracle (bf16 operands, fp32 accumulation).
  * teacher-forced decoder logits: max abs error <= 1.5 % of the largest |logit| against the fp32 oracle.
  * greedy / beam ids on the "lively" weights (Gaussian-like logits, margins down to 1e-3): identical to the storage-rounding
    oracle, except that a window may diverge at a step where the oracle's own top-2 margin is below a DERIVED noise bound:
    8 sigma of the difference of two logits, sigma = the RMS error of the engine's teacher-forced logits against the same
    oracle measured in the same session (near_tie_bound below; ~2e-3 with fp16 storage).  Divergences are logged with their
    margin.  The literal bar - no exemption at all, >= 99 % of >= 128 windows - is tests/test_gpu_parity.py.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
_BOUNDS = {}


def near_tie_bound(which, fx):
    """8 x sqrt(2) x RMS(engine logits - rounding-oracle logits): the margin below which a flipped argmax is noise."""
    if which not in _BOUNDS:
        dims, tok, sd, eng, mel, orc, emu = fx
        enc = eng.encode(mel.cuda())
        toks = np.random.default_rng(5).integers(0, min(dims.vocab, tok.eot), size=(mel.shape[0], 12)).astype(np.int32)
        got = eng.decoder_logits(enc, toks).cpu()
        with torch.no_grad():
            ref = emu.decode(torch.from_numpy(toks).long(), 0, emu.cross_kv(enc.float().cpu()), emu.new_cache())
        rms = (got - ref).pow(2).mean().sqrt().item()
        _BOUNDS[which] = 8.0 * (2.0 ** 0.5) * rms
        print(f"[near-tie bound {which}] logit rms error {rms:.2e} -> bound {_BOUNDS[which]:.2e} (logit std {ref.std().item():.2f})")
    return _BOUNDS[which]


@pytest.fixture(scope="module")
def small():
    from manual_whisper_b200.config import custom_dims, scaled_tokens
    from manual_whisper_b200.weights import random_init
    from manual_whisper_b200.engine import Engine
    from oracle.model import OracleWhisper
    dims = custom_dims("test-small", 80, 128, 2, 2, 2, 512, 2048, n_audio_ctx=200, n_text_ctx=64)
    sd = random_init(dims, seed=21, scheme="lively")
    eng = Engine(dims, sd, 0, max_batch=4, max_beam=5)
    g = torch.Generator().manual_seed(9)
    mel = (torch.randn(4, 80, 400, generator=g) * 0.5).clamp(-1.5, 1.5)
    return dims, scaled_tokens(2048), sd, eng, mel, OracleWhisper(dims, sd), OracleWhisper(dims, sd, emulate=True)


@pytest.fixture(scope="module")
def tiny():
    from manual_whisper_b200.config import model_dims, special_tokens
    from manual_whisper_b200.weights import random_init
    from manual_whisper_b200.engine import Engine
    from oracle.model import OracleWhisper
    dims = model_dims("tiny")
    sd = random_init(dims, seed=1234, scheme="lively")
    eng = Engine(dims, sd, 0, max_batch=2, max_beam=1)
    g = torch.Generator().manual_seed(3)
    mel = (torch.randn(2, 80, 3000, generator=g) * 0.5).clamp(-1.5, 1.5)
    return dims, special_tokens(dims.vocab), sd, eng, mel, OracleWhisper(dims, sd), OracleWhisper(dims, sd, emulate=True)


def rel_l2(a, b):
    return ((a - b).norm() / b.norm()).item()


@pytest.mark.parametrize("which", ["small", "tiny"])
def test_encoder_within_bf16_tolerance(which, request):
    dims, tok, sd, eng, mel, orc, emu = request.getfixturevalue(which)
    got = eng.encode(mel.cuda()).float().cpu()
    with torch.no_grad():
        ref = orc.encode(mel)
    assert got.shape == ref.shape == (mel.shape[0], dims.n_audio_ctx, dims.d_model)
    assert rel_l2(got, ref) <= 2e-2
    # a batch of one gives the same rows as the same chunk inside a larger batch (no cross-chunk leakage)
    one = eng.encode(mel[1:2].cuda()).float().cpu()
    assert torch.equal(one[0], got[1])


def test_encode_time_major_entry_point_equals_encode(small):
    dims, tok, sd, eng, mel, orc, emu = small
    t = torch.zeros(mel.shape[0], 402, 80, dtype=eng.h16, device="cuda")
    t[:, 1:401] = mel.cuda().transpose(1, 2).to(eng.h16)
    assert torch.equal(eng.encode_time_major(t), eng.encode(mel.cuda()))


@pytest.mark.parametrize("which", ["small", "tiny"])
def test_teacher_forced_logits(which, request):
    dims, tok, sd, eng, mel, orc, emu = request.getfixturevalue(which)
    enc = eng.encode(mel.cuda())
    rng = np.random.default_rng(1)
    toks = rng.integers(0, dims.vocab, size=(mel.shape[0], 10)).astype(np.int32)
    got = eng.decoder_logits(enc, toks).cpu()
    with torch.no_grad():
        ref = orc.decode(torch.from_numpy(toks).long(), 0, orc.cross_kv(enc.float().cpu()), orc.new_cache())
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= 1.5e-2 * ref.abs().max().item()


def _compare_ids(got, ref_results, oracle_trace=None):
    report = []
    for b, (g, r) in enumerate(zip(got, ref_results)):
        a, c = g.sequences_ids[0], r.sequences_ids[0]
        k = next((i for i in range(min(len(a), len(c))) if a[i] != c[i]), None)
        if k is None and len(a) == len(c):
            report.append((b, "identical", None))
            continue
        k = min(len(a), len(c)) if k is None else k
        margin = None
        if oracle_trace is not None and k < len(oracle_trace):
            top = oracle_trace[k][b].topk(2).values
            margin = (top[0] - top[1]).item()
        report.append((b, f"diverges@{k}", margin))
    return report


@pytest.mark.parametrize("which", ["small", "tiny"])
@pytest.mark.parametrize("with_ts", [False, True])
def test_greedy_ids(which, with_ts, request):
    from oracle.generate import generate, GenOptions
    dims, tok, sd, eng, mel, orc, emu = request.getfixturevalue(which)
    enc = eng.encode(mel.cuda())
    prompt = [tok.sot, tok.sot + 1, tok.transcribe] + ([] if with_ts else [tok.no_timestamps])
    got = eng.generate(enc, prompt, tok, beam_size=1, max_length=dims.n_text_ctx)
    with torch.no_grad():
        ref, trace = generate(emu, enc.float().cpu(), prompt, tok, GenOptions(beam_size=1, max_length=dims.n_text_ctx), return_trace=True)
    rep = _compare_ids(got, ref, trace)
    print(f"[greedy {which} ts={with_ts}] {rep}")
    bound = near_tie_bound(which, request.getfixturevalue(which))
    for b, status, margin in rep:
        assert status == "identical" or (margin is not None and margin < bound), (b, status, margin, bound)
    n_new = dims.n_text_ctx // 2
    assert all(len(g.sequences_ids[0]) <= n_new for g in got)
    if with_ts:
        for g in got:
            ids = g.sequences_ids[0]
            ts = [t for t in ids if t >= tok.timestamp_begin]
            assert ids[0] >= tok.timestamp_begin and ids[0] <= tok.timestamp_begin + 50 and ts == sorted(ts)
    for g, r in zip(got, ref):
        if g.sequences_ids[0] == r.sequences_ids[0]:
            assert abs(g.scores[0] - r.scores[0]) < 2e-2


def _oracle_score(model, enc1, prompt, ids, tok, n_new, length_penalty=1.0):
    """Length-normalised log-probability the ORACLE assigns to `ids` (rules applied at every step)."""
    from oracle.generate import apply_rules, expand_suppress
    with_ts = prompt[-1] != tok.no_timestamps
    sup = expand_suppress(tok, [-1], with_ts)
    ended = len(ids) < n_new
    seq = list(ids) + ([tok.eot] if ended else [])
    inp = torch.tensor([prompt + seq[:-1]])
    with torch.no_grad():
        logits = model.decode(inp, 0, model.cross_kv(enc1), model.new_cache())[0]
    total = 0.0
    for i, t in enumerate(seq):
        row = apply_rules(logits[len(prompt) - 1 + i][None], [seq[:i]], tok, sup, tok.suppress_ids_begin, with_ts, 50)
        total += float(torch.log_softmax(row.float(), -1)[0, t])
    return total / (len(seq) ** length_penalty)


@pytest.mark.parametrize("with_ts", [False, True])
@pytest.mark.parametrize("beam,patience", [(5, 1.0), (3, 2.0)])
def test_beam_ids(small, with_ts, beam, patience):
    from oracle.generate import generate, GenOptions
    dims, tok, sd, eng, mel, orc, emu = small
    enc = eng.encode(mel.cuda())
    prompt = [tok.sot, tok.sot + 1, tok.transcribe] + ([] if with_ts else [tok.no_timestamps])
    got = eng.generate(enc, prompt, tok, beam_size=beam, patience=patience, max_length=dims.n_text_ctx, num_hypotheses=beam)
    with torch.no_grad():
        ref = generate(emu, enc.float().cpu(), prompt, tok, GenOptions(beam_size=beam, patience=patience,
                                                                     max_length=dims.n_text_ctx, num_hypotheses=beam))
    same = [g.sequences_ids[0] == r.sequences_ids[0] for g, r in zip(got, ref)]
    print(f"[beam{beam} p={patience} ts={with_ts}] identical {sum(same)}/{len(same)} scores",
          [(round(g.scores[0], 4), round(r.scores[0], 4)) for g, r in zip(got, ref)])
    # beam search compounds the near-ties of random-init weights: a window may end on a different but equally good
    # hypothesis.  Required: the engine's own score agrees with the oracle's best score, and the engine's hypothesis
    # RE-SCORED BY THE ORACLE is as good as the oracle's best one (so it is a legitimate winner, not an error).
    n_new = dims.n_text_ctx // 2 if len(prompt) <= dims.n_text_ctx // 2 else dims.n_text_ctx - len(prompt)
    for b, (g, r) in enumerate(zip(got, ref)):
        assert abs(g.scores[0] - r.scores[0]) < 3e-2
        assert g.scores == sorted(g.scores, reverse=True)
        if not same[b]:
            rescored = _oracle_score(emu, enc.float().cpu()[b:b + 1], prompt, g.sequences_ids[0], tok, n_new)
            print(f"  window {b}: different hypothesis; oracle re-score {rescored:.4f} vs oracle best {r.scores[0]:.4f}")
            assert rescored >= r.scores[0] - 3e-2
    assert sum(same) >= len(same) // 2


def test_eot_and_forced_eot_and_long_prompt(small):
    from oracle.generate import generate, GenOptions
    import dataclasses
    dims, tok, sd, eng, mel, orc, emu = small
    enc = eng.encode(mel.cuda())
    prompt = [tok.sot, tok.sot + 1, tok.transcribe, tok.no_timestamps]
    base = eng.generate(enc, prompt, tok, beam_size=1, max_length=dims.n_text_ctx)
    # make a frequently generated id play <eot>: sequences must stop there, eot excluded, on both sides
    ids = base[0].sequences_ids[0]
    fake_eot = ids[3]
    tok2 = dataclasses.replace(tok, eot=fake_eot)
    got = eng.generate(enc, prompt, tok2, beam_size=1, max_length=dims.n_text_ctx, suppress_tokens=[], suppress_blank=False)
    with torch.no_grad():
        ref = generate(emu, enc.float().cpu(), prompt, tok2, GenOptions(beam_size=1, max_length=dims.n_text_ctx,
                                                                       suppress_tokens=[], suppress_blank=False))
    assert all(fake_eot not in g.sequences_ids[0] for g in got)
    assert [g.sequences_ids[0] for g in got][0] == ref[0].sequences_ids[0]
    assert len(got[0].sequences_ids[0]) < len(ids)
    forced = eng.generate(enc, prompt, tok, beam_size=1, max_length=dims.n_text_ctx, forced_eot_len=5)
    assert all(len(g.sequences_ids[0]) == 5 for g in forced)
    assert forced[0].sequences_ids[0] == ids[:5]
    # long prompt (initial_prompt path): [sot_prev] + 20 ids + sot sequence
    rng = np.random.default_rng(2)
    lp = [tok.sot_prev] + rng.integers(300, 1500, size=20).tolist() + prompt
    got = eng.generate(enc, lp, tok, beam_size=1, max_length=dims.n_text_ctx)
    with torch.no_grad():
        ref, trace = generate(emu, enc.float().cpu(), lp, tok, GenOptions(beam_size=1, max_length=dims.n_text_ctx), return_trace=True)
    for b, status, margin in _compare_ids(got, ref, trace):
        assert status == "identical" or (margin is not None and margin < near_tie_bound("small", small)), (b, status, margin)
    assert all(len(g.sequences_ids[0]) <= min(dims.n_text_ctx // 2, dims.n_text_ctx - len(lp)) for g in got)


def test_generate_argument_errors(small):
    dims, tok, sd, eng, mel, orc, emu = small
    enc = eng.encode(mel.cuda())
    with pytest.raises(ValueError, match="beam_size"):
        eng.generate(enc, [tok.sot], tok, beam_size=7)
    with pytest.raises(ValueError, match="vocabulary"):
        eng.generate(enc, [tok.vocab + 5], tok, beam_size=1, max_length=dims.n_text_ctx)
    with pytest.raises(ValueError, match="max_length"):
        eng.generate(enc, [tok.sot], tok, beam_size=1, max_length=4096)
    with pytest.raises(ValueError, match="prompt"):
        eng.generate(enc, [], tok, beam_size=1)


def test_detect_language_matches_oracle(small):
    dims, tok, sd, eng, mel, orc, emu = small
    enc = eng.encode(mel.cuda())
    probs = eng.detect_language(enc, tok)
    with torch.no_grad():
        lg = emu.decode(torch.full((mel.shape[0], 1), tok.sot), 0, emu.cross_kv(enc.float().cpu()), emu.new_cache())[:, 0]
    ref = torch.softmax(lg[:, tok.sot + 1: tok.sot + 1 + tok.n_langs], dim=-1).numpy()
    assert probs.shape == ref.shape and np.abs(probs - ref).max() < 2e-2 and np.allclose(probs.sum(1), 1.0, atol=1e-5)


@pytest.mark.parametrize("beam", [1, 3])
def test_long_prompt_batched_prefill_equals_stepwise_oracle(small, beam):
    """Prompts longer than 4 tokens go through the batched (tensor-core) prefill; the oracle prefills in one masked pass."""
    from oracle.generate import generate, GenOptions
    dims, tok, sd, eng, mel, orc, emu = small
    enc = eng.encode(mel.cuda())
    rng = np.random.default_rng(11)
    lp = [tok.sot_prev] + rng.integers(300, 1500, size=25).tolist() + [tok.sot, tok.sot + 2, tok.transcribe, tok.no_timestamps]
    got = eng.generate(enc, lp, tok, beam_size=beam, max_length=dims.n_text_ctx)
    n_new = dims.n_text_ctx - len(lp) if len(lp) > dims.n_text_ctx // 2 else dims.n_text_ctx // 2
    assert all(len(g.sequences_ids[0]) <= n_new for g in got)
    if beam == 1:
        with torch.no_grad():
            ref, trace = generate(emu, enc.float().cpu(), lp, tok, GenOptions(beam_size=1, max_length=dims.n_text_ctx), return_trace=True)
        for b, status, margin in _compare_ids(got, ref, trace):
            assert status == "identical" or (margin is not None and margin < near_tie_bound("small", small)), (b, status, margin)
        return
    with torch.no_grad():
        ref = generate(emu, enc.float().cpu(), lp, tok, GenOptions(beam_size=beam, max_length=dims.n_text_ctx))
    for b, (g, r) in enumerate(zip(got, ref)):
        if g.sequences_ids[0] == r.sequences_ids[0]:
            assert abs(g.scores[0] - r.scores[0]) < 3e-2
        else:
            rescored = _oracle_score(emu, enc.float().cpu()[b:b + 1], lp, g.sequences_ids[0], tok, n_new)
            print(f"  window {b}: different ids; oracle re-score {rescored:.4f} vs oracle best {r.scores[0]:.4f}")
            assert rescored >= r.scores[0] - 6e-2      # pruning at a near-tie may end on a slightly worse hypothesis


def test_batched_prefill_matches_stepwise_prefill(small, monkeypatch):
    """Engine against engine: the one-pass tensor-core prefill and the token-by-token prefill leave the same state."""
    dims, tok, sd, eng, mel, orc, emu = small
    enc = eng.encode(mel.cuda())
    rng = np.random.default_rng(12)
    lp = [tok.sot_prev] + rng.integers(300, 1500, size=20).tolist() + [tok.sot, tok.sot + 1, tok.transcribe, tok.no_timestamps]
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("MW_STEPWISE_PREFILL", mode)
        res[mode] = {beam: eng.generate(enc, lp, tok, beam_size=beam, max_length=dims.n_text_ctx) for beam in (1, 5)}
    for beam in (1, 5):
        same = [a.sequences_ids[0] == b.sequences_ids[0] for a, b in zip(res["0"][beam], res["1"][beam])]
        prefix = [next((i for i, (x, y) in enumerate(zip(a.sequences_ids[0], b.sequences_ids[0])) if x != y), len(a.sequences_ids[0]))
                  for a, b in zip(res["0"][beam], res["1"][beam])]
        print(f"  beam {beam}: identical {sum(same)}/{len(same)}, common prefixes {prefix}")
        assert sum(same) >= len(same) - 1 and all(p >= 3 for p in prefix)
        for a, b in zip(res["0"][beam], res["1"][beam]):
            assert abs(a.scores[0] - b.scores[0]) < 3e-2


@pytest.mark.parametrize("which", ["small", "tiny"])
def test_solo_mode_decodes_the_same_ids(which, request):
    """mw_set_solo folds LayerNorm into the projections that consume it (same lane mapping, summation order and rounding as
    the stand-alone kernel): greedy and beam ids and scores must not move by a bit."""
    dims, tok, sd, eng, mel, orc, emu = request.getfixturevalue(which)
    enc = eng.encode(mel.cuda())
    prompt = [tok.sot, tok.sot + 1, tok.transcribe, tok.no_timestamps]
    beams = (1, 5) if which == "small" else (1,)          # the tiny fixture's engine is built for greedy only
    res = {}
    try:
        for solo in (False, True):
            eng.set_solo(solo)
            res[solo] = {beam: eng.generate(enc, prompt, tok, beam_size=beam, max_length=64) for beam in beams}
    finally:
        eng.set_solo(False)
    for beam in beams:
        for a, b in zip(res[False][beam], res[True][beam]):
            assert a.sequences_ids[0] == b.sequences_ids[0]
            assert a.scores[0] == b.scores[0]


@pytest.fixture(scope="module")
def wide():
    """The test-small dims with 100 windows: a step of >= 96 rows runs every projection on the tcgen05 decode GEMM (greedy) and
    the vocabulary projection on it in beam search (5 beams x 20 windows)."""
    from manual_whisper_b200.config import custom_dims, scaled_tokens
    from manual_whisper_b200.weights import random_init
    from manual_whisper_b200.engine import Engine
    from oracle.model import OracleWhisper
    dims = custom_dims("test-small", 80, 128, 2, 2, 2, 512, 2048, n_audio_ctx=200, n_text_ctx=64)
    sd = random_init(dims, seed=23, scheme="lively")
    eng = Engine(dims, sd, 0, max_batch=100, max_beam=5)
    g = torch.Generator().manual_seed(19)
    mel = (torch.randn(100, 80, 400, generator=g) * 0.5).clamp(-1.5, 1.5)
    return dims, scaled_tokens(2048), sd, eng, mel, OracleWhisper(dims, sd), OracleWhisper(dims, sd, emulate=True)


def test_teacher_forced_logits_at_100_rows(wide):
    """100 rows against the oracle, and against the same windows decoded 32 at a time (the mma.sync projections).  The two
    engine paths sum in different orders, so their 16-bit activations round differently here and there, and they differ by
    about what either differs from the fp32 oracle (B200: 9.4e-4 and 1.05e-3 of the largest |logit|).  The engine-vs-engine
    bound is 2^-8 of the largest |logit|, a quarter of the bound against the oracle."""
    dims, tok, sd, eng, mel, orc, emu = wide
    enc = eng.encode(mel.cuda())
    toks = np.random.default_rng(4).integers(0, dims.vocab, size=(mel.shape[0], 10)).astype(np.int32)
    got = eng.decoder_logits(enc, toks).cpu()
    with torch.no_grad():
        ref = orc.decode(torch.from_numpy(toks).long(), 0, orc.cross_kv(enc.float().cpu()), orc.new_cache())
    top = ref.abs().max().item()
    print(f"[100 rows] max |engine - oracle| = {(got - ref).abs().max().item() / top:.2e} of max |logit|")
    assert (got - ref).abs().max().item() <= 1.5e-2 * top
    parts = torch.cat([eng.decoder_logits(enc[i:i + 32], toks[i:i + 32]).cpu() for i in range(0, mel.shape[0], 32)])
    diff = (got - parts).abs().max().item()
    print(f"[100 rows] max |100 rows - 32-row batches| = {diff / top:.2e} of max |logit|")
    assert diff <= 2.0 ** -8 * top


def test_greedy_ids_at_100_rows(wide):
    from oracle.generate import generate, GenOptions
    dims, tok, sd, eng, mel, orc, emu = wide
    enc = eng.encode(mel.cuda())
    prompt = [tok.sot, tok.sot + 1, tok.transcribe, tok.no_timestamps]
    got = eng.generate(enc, prompt, tok, beam_size=1, max_length=dims.n_text_ctx)
    with torch.no_grad():
        ref, trace = generate(emu, enc.float().cpu(), prompt, tok, GenOptions(beam_size=1, max_length=dims.n_text_ctx), return_trace=True)
    rep = _compare_ids(got, ref, trace)
    bound = near_tie_bound("wide", wide)
    print(f"[greedy 100 rows] identical {sum(s == 'identical' for _, s, _ in rep)}/{len(rep)}")
    for b, status, margin in rep:
        assert status == "identical" or (margin is not None and margin < bound), (b, status, margin, bound)


def test_beam_ids_at_100_rows(wide):
    """Beam 5 x 20 windows: the layer projections on mma.sync, the vocabulary projection on the decode GEMM."""
    from oracle.generate import generate, GenOptions
    dims, tok, sd, eng, mel, orc, emu = wide
    enc = eng.encode(mel[:20].cuda())
    prompt = [tok.sot, tok.sot + 1, tok.transcribe, tok.no_timestamps]
    got = eng.generate(enc, prompt, tok, beam_size=5, max_length=dims.n_text_ctx, num_hypotheses=5)
    with torch.no_grad():
        ref = generate(emu, enc.float().cpu(), prompt, tok, GenOptions(beam_size=5, max_length=dims.n_text_ctx, num_hypotheses=5))
    same = [g.sequences_ids[0] == r.sequences_ids[0] for g, r in zip(got, ref)]
    print(f"[beam5 x 20] identical {sum(same)}/{len(same)}")
    n_new = dims.n_text_ctx // 2
    for b, (g, r) in enumerate(zip(got, ref)):
        assert abs(g.scores[0] - r.scores[0]) < 3e-2
        assert g.scores == sorted(g.scores, reverse=True)
        if not same[b]:
            rescored = _oracle_score(emu, enc.float().cpu()[b:b + 1], prompt, g.sequences_ids[0], tok, n_new)
            print(f"  window {b}: different hypothesis; oracle re-score {rescored:.4f} vs oracle best {r.scores[0]:.4f}")
            assert rescored >= r.scores[0] - 3e-2
    assert sum(same) >= len(same) // 2
