"""The decode step's kernels (csrc/decoder.cu) pinned one by one against float64 references, through the test entry points
mw_step_*_h16 (include/mw_b200.h), on every launch path the step can take.

References are computed in float64 on the device from the exact 16-bit inputs the kernel reads.  Every element is held to a
bound scaled to THAT element (never to the largest output):
  * projections: |got - ref| <= 2^-18 sqrt(K) (|X| |W|^T)[r,n] + 2^-22 (|bias| + |resid| + |ref|), x 1.2 through GELU
    (max |gelu'| < 1.13), plus half an ulp of the storage type for 16-bit output.  fp32 accumulation of K products errs by
    about 2^-24 sqrt(K) (|X| |W|^T) (random rounding), so the bound has a 64x margin; for K = 5120 it is still ~1 % of a
    typical |ref|, while losing one 32-wide block of K moves an output by ~8 % of |ref|.
  * attention: |got - ref| <= half-ulp(|ref|) + 2^-14 max_j |v_j| per (row, head, column): scores and probabilities are
    fp32 (__expf is accurate to a few ulp), so what is left is the rounding of the 16-bit output - plus, for scores of large
    magnitude, the fp32 rounding of the scores themselves (_attend).
Rows past R are NaN sentinels and must stay NaN.  Paths that the code says give the same bits are compared bit for bit.
"""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
GREEDY, BEAM, GREEDY_SOLO, BEAM_SOLO, ROWS16_WT1, ROWS16_WT2, KHALF_WT1, KHALF_WT2, GENERIC, LN_FUSED, LN_SEPARATE = range(11)
PATH_NAMES = ["greedy", "beam", "greedy_solo", "beam_solo", "rows16_wt1", "rows16_wt2", "khalf_wt1", "khalf_wt2", "generic",
              "ln_fused", "ln_separate"]
GELU, F32 = 1, 2
ROWS = [1, 17, 31, 32, 33, 80, 160, 256]       # rows on the mma.sync paths
DG_ROWS = [95, 96, 128, 256]                   # rows through the greedy routing (tcgen05 decode GEMM from 96)
INDEP_ROWS = [1, 17, 32, 33, 80]               # a row's bits must not depend on how many rows share the launch

# the tuned-kernel table of skinny_gemm (MW_SK): K -> warps per CTA; K = KB * NW * 32
SK_WARPS = {128: 4, 384: 4, 256: 8, 512: 8, 768: 8, 1024: 8, 1280: 8, 1536: 8, 2048: 16, 3072: 16, 4096: 16, 5120: 16}


def has_rows16_wt2(K):
    return K in SK_WARPS and SK_WARPS[K] <= 8 and K // (SK_WARPS[K] * 32) <= 5


def has_khalf(K):
    return K in SK_WARPS and SK_WARPS[K] == 16


# (d_model, ffn, vocab) of the step's shapes: tiny, base, small, medium, large-v3, the test-small dims, and two widths without a
# tuned kernel (the generic fallback: d = 640, ffn = 2560) or with only the 256 entry
MODELS = {"tiny": (384, 1536, 51865), "base": (512, 2048, 51865), "small": (768, 3072, 51865), "medium": (1024, 4096, 51865),
          "large-v3": (1280, 5120, 51866), "test-small": (128, 512, 2048), "d256": (256, 1024, 2048),
          "d640": (640, 2560, 4096)}


def step_projections(d, ffn, vocab):
    """(name, N, K, flags, residual, layernorm) of every projection of one decode step."""
    return [("qkv", 3 * d, d, 0, False, True), ("out", d, d, F32, True, False), ("cross_q", d, d, 0, False, True),
            ("fc1", ffn, d, GELU, False, True), ("fc2", d, ffn, F32, True, False), ("logits", vocab, d, F32, False, True)]


PROJ_CASES = [(m, *p) for m, dims in MODELS.items() for p in step_projections(*dims)]
PROJ_CASES += [("ragged", "n%32=1", 32 * 65 + 1, 512, F32, True, False), ("ragged", "n%32=17-gelu", 32 * 40 + 17, 1280, GELU, False, False),
               ("ragged", "n%32=17-k5120", 32 * 40 + 17, 5120, 0, False, False)]
LN_CASES = [c for c in PROJ_CASES if c[6]]


def _h16():
    from manual_whisper_b200 import _lib
    return _lib.storage_dtype()


def _half_ulp():
    return 2.0 ** -11 if _h16() == torch.float16 else 2.0 ** -8


@pytest.fixture(scope="module")
def lib():
    from manual_whisper_b200 import _lib
    return _lib.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _report(what, worst):
    print(f"[{what}] worst |err| / bound = {worst:.3f}")


def _check_bound(got, ref, bound, what):
    """Element-wise |got - ref| <= bound (NaN fails); returns the worst ratio."""
    err = (got.double() - ref).abs()
    ratio = err / bound
    worst = ratio.max().item() if ratio.numel() else 0.0
    bad = ~(err <= bound)
    if bad.any():
        idx = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} elements out of bound; first at {idx}: got {got[tuple(idx)].item()!r} "
                             f"ref {ref[tuple(idx)].item()!r} bound {bound[tuple(idx)].item():.3e} (worst ratio {worst:.2f})")
    return worst


# ------------------------------------------------------------------------------------------------ projections
class Proj:
    """Seeded inputs of one projection shape with room for 256 rows, and its float64 reference."""

    def __init__(self, N, K, flags, resid, seed):
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.N, self.K, self.flags = N, K, flags
        self.x = (torch.randn(256, K, device=DEV, generator=g) * 0.5).to(_h16())
        self.w = (torch.randn(N, K, device=DEV, generator=g) * 0.05).to(_h16())
        self.bias = torch.randn(N, device=DEV, generator=g) * 0.1
        self.resid = torch.randn(256, N, device=DEV, generator=g) if resid else None
        self.out_dtype = torch.float32 if flags & F32 else _h16()

    def reference(self, x16):
        """float64 reference and per-element bound for the 16-bit operand x16 [R, K]."""
        xd, wd = x16.double(), self.w.double()
        pre = xd @ wd.t() + self.bias.double()
        mag = x16.double().abs() @ wd.abs().t()
        bound = 2.0 ** -18 * self.K ** 0.5 * mag + 2.0 ** -22 * (self.bias.double().abs() + pre.abs())
        ref = pre
        if self.flags & GELU:
            ref = 0.5 * pre * (1.0 + torch.erf(pre / 2.0 ** 0.5))
            bound = bound * 1.2
        if self.resid is not None:
            r = self.resid[: x16.shape[0]].double()
            ref = ref + r
            bound = bound + 2.0 ** -22 * r.abs()
        bound = bound + 2.0 ** -22 * ref.abs()
        if not self.flags & F32:
            bound = bound + _half_ulp() * ref.abs() + 2.0 ** -25
        return ref, bound

    def run(self, lib, R, path, x16=None, ln=None):
        """out with two NaN sentinel rows past R; ln = (x_f32, gamma, beta, scratch h16) runs the LayerNorm paths."""
        out = torch.full((R + 2, self.N), float("nan"), device=DEV, dtype=self.out_dtype)
        resid = self.resid[:R].contiguous() if self.resid is not None else None
        if ln is None:
            args = (_ptr(self.x[:R] if x16 is None else x16), None, None, None)
        else:
            xf, gam, bet, scratch = ln
            args = (_ptr(scratch), _ptr(xf), _ptr(gam), _ptr(bet))
        from manual_whisper_b200 import _lib
        _lib.check(lib.mw_step_projection_h16(*args, _ptr(self.w), _ptr(self.bias), _ptr(resid), _ptr(out), R, self.N, self.K,
                                              self.flags, path, _stream()), f"mw_step_projection_h16 path {PATH_NAMES[path]}")
        torch.cuda.synchronize()
        assert torch.isnan(out[R:].float()).all(), f"path {PATH_NAMES[path]} R={R}: rows past R were written"
        return out[:R]


def _mma_paths(K):
    paths = [BEAM, BEAM_SOLO, GENERIC]
    if K in SK_WARPS:
        paths.append(ROWS16_WT1)
    if has_rows16_wt2(K):
        paths.append(ROWS16_WT2)
    if has_khalf(K):
        paths += [KHALF_WT1, KHALF_WT2]
    return paths


@pytest.mark.parametrize("model,name,N,K,flags,resid,ln", PROJ_CASES, ids=[f"{c[0]}-{c[1]}" for c in PROJ_CASES])
def test_projection(lib, model, name, N, K, flags, resid, ln):
    """Every projection kernel the step can run for this (N, K, flags), at ragged row counts, against float64."""
    p = Proj(N, K, flags, resid, seed=N * 31 + K)
    ref, bound = p.reference(p.x)
    worst = 0.0
    full = {}
    for path in _mma_paths(K):
        for R in ROWS:
            got = p.run(lib, R, path)
            worst = max(worst, _check_bound(got, ref[:R], bound[:R], f"{model} {name} {PATH_NAMES[path]} R={R}"))
            if R == 256:
                full[path] = got
        again = p.run(lib, 256, path)
        assert torch.equal(again, full[path]), f"{PATH_NAMES[path]}: two runs differ"
        for R in INDEP_ROWS:
            assert torch.equal(p.run(lib, R, path), full[path][:R]), f"{PATH_NAMES[path]}: rows depend on R={R}"
    # the same-bits claims of the code
    if has_rows16_wt2(K):
        assert torch.equal(full[ROWS16_WT1], full[ROWS16_WT2]), "rows16: one and two weight tiles differ"
        assert torch.equal(full[BEAM], full[ROWS16_WT2])
    if has_khalf(K):
        assert torch.equal(full[KHALF_WT1], full[KHALF_WT2]), "K-halved kernel: one and two weight tiles differ"
        assert torch.equal(full[BEAM], full[KHALF_WT2]) and torch.equal(full[BEAM_SOLO], full[KHALF_WT1])
    if K not in SK_WARPS:
        assert torch.equal(full[BEAM], full[GENERIC])
    # the greedy routing: mma.sync below 96 rows, the tcgen05 decode GEMM from 96 rows on
    dg = {}
    for R in DG_ROWS:
        got = p.run(lib, R, GREEDY)
        worst = max(worst, _check_bound(got, ref[:R], bound[:R], f"{model} {name} greedy R={R}"))
        if R < 96:
            assert torch.equal(got, full[BEAM][:R])
        dg[R] = got
    assert torch.equal(p.run(lib, 256, GREEDY), dg[256]), "decode GEMM: two runs differ"
    for R in (96, 128):
        assert torch.equal(dg[R], dg[256][:R]), f"decode GEMM: rows depend on R={R}"
    _report(f"{model} {name} N={N} K={K}", worst)


def _layernorm_ref(xf, gam, bet):
    xd = xf.double()
    mu = xd.mean(-1, keepdim=True)
    var = ((xd - mu) ** 2).mean(-1, keepdim=True)
    return (xd - mu) / torch.sqrt(var + 1e-5) * gam.double() + bet.double()


@pytest.mark.parametrize("model,name,N,K,flags,resid,ln", LN_CASES, ids=[f"{c[0]}-{c[1]}" for c in LN_CASES])
def test_layernorm_projection(lib, model, name, N, K, flags, resid, ln):
    """LayerNorm + projection: the stand-alone LayerNorm and the fused kernel give the same bits; both against float64."""
    p = Proj(N, K, flags, False, seed=N * 17 + K)
    g = torch.Generator(device=DEV).manual_seed(K)
    xf = torch.randn(256, K, device=DEV, generator=g) * 3 + 1
    gam = 1 + 0.2 * torch.randn(K, device=DEV, generator=g)
    bet = 0.2 * torch.randn(K, device=DEV, generator=g)
    fused = K in SK_WARPS and has_rows16_wt2(K) and not flags & F32
    worst = 0.0
    sep = {}

    def run(R, path):
        scratch = torch.full((R, K), float("nan"), device=DEV, dtype=_h16())
        got = p.run(lib, R, path, ln=(xf[:R].contiguous(), gam, bet, scratch))
        return got, scratch

    for R in ROWS + [95, 96, 128]:
        got, scratch = run(R, LN_SEPARATE)
        # the 16-bit operand the projection read: LayerNorm of x to half an ulp
        lref = _layernorm_ref(xf[:R], gam, bet)
        _check_bound(scratch, lref, _half_ulp() * lref.abs() + 2.0 ** -18 * (gam.double().abs() + 1) + 2.0 ** -25,
                     f"{model} {name} LayerNorm R={R}")
        ref, bound = p.reference(scratch)
        worst = max(worst, _check_bound(got, ref, bound, f"{model} {name} ln_separate R={R}"))
        sep[R] = got
        assert torch.equal(run(R, BEAM)[0], got)
        assert torch.equal(run(R, BEAM_SOLO)[0], got), "solo (fused LayerNorm) and separate LayerNorm differ"
        if fused:
            assert torch.equal(run(R, LN_FUSED)[0], got), "fused LayerNorm projection and LayerNorm + projection differ"
        gr, gscratch = run(R, GREEDY)
        if R < 96:
            assert torch.equal(gr, got)
        else:        # LayerNorm, then the tcgen05 decode GEMM
            ref, bound = p.reference(gscratch)
            worst = max(worst, _check_bound(gr, ref, bound, f"{model} {name} greedy R={R}"))
            assert torch.equal(run(R, GREEDY_SOLO)[0], gr)
    for R in INDEP_ROWS:
        assert torch.equal(sep[R], sep[256][:R])
        if fused:
            assert torch.equal(run(R, LN_FUSED)[0], sep[256][:R])
    if not fused:
        with pytest.raises(RuntimeError, match="no fused"):
            run(32, LN_FUSED)
    _report(f"{model} {name} LN N={N} K={K}", worst)


def test_forced_path_missing_for_k_is_an_error(lib):
    p = Proj(64, 640, 0, False, seed=1)
    for path in (ROWS16_WT1, ROWS16_WT2, KHALF_WT1, KHALF_WT2):
        with pytest.raises(RuntimeError, match="K=640"):
            p.run(lib, 32, path)
    q = Proj(64, 1536, 0, False, seed=2)
    with pytest.raises(RuntimeError, match="two-tile"):
        q.run(lib, 32, ROWS16_WT2)
    assert lib.mw_step_projection_h16(_ptr(q.x), None, None, None, _ptr(q.w), None, None, _ptr(q.x), 32, 64, 1536, 0, KHALF_WT2,
                                      _stream()) == 3
    assert b"K-halved" in lib.mw_last_error()


# ------------------------------------------------------------------------------------------------ attention references
def _score_slack(q, k):
    """Largest sum_i |q_i k_i| / 8 over the keys (q [..., 64], k [..., n, 64] -> [..., 1]): the scores are fp32 sums of 64
    products, each off by up to ~2^-21 of this."""
    return (q.double().abs().unsqueeze(-2) @ k.double().abs().transpose(-1, -2)).squeeze(-2).amax(dim=-1, keepdim=True) / 8.0


def _attend(q, k, v):
    """float64 softmax(q k^T / 8) v and its bound: q [..., 64], k/v [..., n, 64] (16-bit values, exact in float64).
    Besides the bound of the module docstring, an error e in every score moves the output by up to 2 e max|v|: with scores of
    +-60 (sum |q_i k_i| / 8 ~ 300) that is 2^-20 x 300 max|v|, above 2^-14 max|v|; with random inputs it is ~2^-18 max|v|."""
    s = (q.double().unsqueeze(-2) @ k.double().transpose(-1, -2)).squeeze(-2) / 8.0
    pr = torch.softmax(s, dim=-1)
    ref = (pr.unsqueeze(-2) @ v.double()).squeeze(-2)
    vmax = v.double().abs().amax(dim=-2)
    bound = _half_ulp() * ref.abs() + (2.0 ** -14 + 2.0 ** -20 * _score_slack(q, k)) * vmax + 2.0 ** -25
    return ref, bound


# ------------------------------------------------------------------------------------------------ self-attention
SELF_POS = [0, 1, 3, 15, 16, 17, 63, 64, 65, 223, 447]


@pytest.mark.parametrize("beam", [False, True], ids=["greedy", "beam5"])
@pytest.mark.parametrize("heads", [6, 20])
def test_self_attention(lib, heads, beam):
    """decode_attn_kernel<true>: append this step's k, v at pos, attend over pos + 1 keys (through the beam index table)."""
    from manual_whisper_b200 import _lib
    d, ctx = heads * 64, 448
    worst = 0.0
    for R in (1, 5, 32):
        g = torch.Generator(device=DEV).manual_seed(heads * 100 + R + 7 * beam)
        kc0 = torch.randn(R, ctx, d, device=DEV, generator=g).to(_h16())
        vc0 = torch.randn(R, ctx, d, device=DEV, generator=g).to(_h16())
        for pos in SELF_POS:
            qkv = torch.randn(R, 3 * d, device=DEV, generator=g).to(_h16())
            kc, vc = kc0.clone(), vc0.clone()
            idx = None
            if beam:     # a random parent row inside each group of 5 beams for every earlier position
                grp = torch.arange(R, device=DEV) // 5 * 5
                size = torch.clamp(R - grp, max=5)
                off = (torch.rand(R, ctx, device=DEV, generator=g) * size[:, None]).long()
                idx = (grp[:, None] + off).to(torch.int32).contiguous()
            out = torch.full((R + 1, d), float("nan"), device=DEV, dtype=_h16())
            _lib.check(lib.mw_step_self_attention_h16(_ptr(qkv), _ptr(kc), _ptr(vc), _ptr(idx), R, heads, ctx, pos, _ptr(out),
                                                      _stream()), "mw_step_self_attention_h16")
            torch.cuda.synchronize()
            q, knew, vnew = qkv.view(R, 3, heads, 64).unbind(1)
            # the only cache change: row r, position pos = this step's k, v
            ek, ev = kc0.clone(), vc0.clone()
            ek[:, pos] = knew.reshape(R, d)
            ev[:, pos] = vnew.reshape(R, d)
            assert torch.equal(kc, ek) and torch.equal(vc, ev), f"R={R} pos={pos}: cache writes"
            rows = torch.arange(R, device=DEV)[:, None].expand(R, pos + 1).clone()
            if idx is not None:
                rows[:, :pos] = idx[:, :pos].long()
            cols = torch.arange(pos + 1, device=DEV)[None].expand(R, pos + 1)
            keys = ek[rows, cols].view(R, pos + 1, heads, 64).transpose(1, 2)       # [R, heads, pos+1, 64]
            vals = ev[rows, cols].view(R, pos + 1, heads, 64).transpose(1, 2)
            ref, bound = _attend(q, keys, vals)
            worst = max(worst, _check_bound(out[:R].view(R, heads, 64), ref, bound, f"self-attention R={R} pos={pos} beam={beam}"))
            assert torch.isnan(out[R:].float()).all()
    _report(f"self-attention heads={heads} beam={beam}", worst)


# ------------------------------------------------------------------------------------------------ batched-prefill attention
@pytest.mark.parametrize("heads", [6, 20])
def test_prefill_attention(lib, heads):
    """decode_attn_kernel<false> as batched_prefill launches it: row (b, p) attends causally over keys 0..p of sequence b."""
    from manual_whisper_b200 import _lib
    d = heads * 64
    worst = 0.0
    for B in (1, 3):
        for P in (4, 5, 31, 64, 223):
            g = torch.Generator(device=DEV).manual_seed(B * 1000 + P + heads)
            qkv = torch.randn(B * P, 3 * d, device=DEV, generator=g).to(_h16())
            out = torch.full((B * P + 1, d), float("nan"), device=DEV, dtype=_h16())
            _lib.check(lib.mw_step_prefill_attention_h16(_ptr(qkv), B, P, heads, _ptr(out), _stream()), "mw_step_prefill_attention_h16")
            torch.cuda.synchronize()
            q, k, v = [t.reshape(B, P, heads, 64).transpose(1, 2).double() for t in qkv.view(B * P, 3, d).unbind(1)]
            s = q @ k.transpose(-1, -2) / 8.0
            s = s.masked_fill(torch.ones(P, P, dtype=torch.bool, device=DEV).triu(1), float("-inf"))
            ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * P, heads, 64)
            vmax = torch.cummax(v.abs(), dim=2).values.transpose(1, 2).reshape(B * P, heads, 64)     # max over the keys seen
            slack = ((q.abs() @ k.abs().transpose(-1, -2)).amax(-1, keepdim=True) / 8.0).transpose(1, 2).reshape(B * P, heads, 1)
            bound = _half_ulp() * ref.abs() + (2.0 ** -14 + 2.0 ** -20 * slack) * vmax + 2.0 ** -25
            worst = max(worst, _check_bound(out[:B * P].view(B * P, heads, 64), ref, bound, f"prefill B={B} P={P}"))
            assert torch.isnan(out[B * P:].float()).all()
    _report(f"prefill heads={heads}", worst)


# ------------------------------------------------------------------------------------------------ cross-attention
CROSS_T = [1, 2, 15, 16, 17, 63, 64, 65, 1499, 1500]
CROSS_G = [(1, 4), (1, 8)] + [(G, 0) for G in range(2, 9)]


def _cross_inputs(mode, B, G, T, heads, g):
    d = heads * 64
    q = torch.randn(B * G, d, device=DEV, generator=g)
    k = torch.randn(B * T, d, device=DEV, generator=g)
    v = torch.randn(B * T, d, device=DEV, generator=g)
    if mode == "increasing":       # score of key j grows with j: the online softmax rescales at every key
        q = torch.ones_like(q)
        s = torch.linspace(-20.0, 40.0, T, device=DEV).repeat(B)
        k = (s / 8.0)[:, None].expand(B * T, d) * (1 + 0.01 * torch.randn(B * T, d, device=DEV, generator=g))
    elif mode == "dominant":       # one key, the last, carries almost all the weight
        k = k.view(B, T, d)
        k[:, -1] = q.view(B, G, d).mean(1) * 3.0
        k = k.reshape(B * T, d)
    elif mode == "large":          # score magnitudes around +-60
        q, k = q * 60.0 ** 0.5, k * 60.0 ** 0.5
    return q.to(_h16()), torch.cat([k, v], dim=1).to(_h16()).contiguous()


@pytest.mark.parametrize("heads", [6, 20])
@pytest.mark.parametrize("mode", ["random", "increasing", "dominant", "large"])
def test_cross_attention(lib, mode, heads):
    """cross_attn_stream_kernel<4|8> (greedy) and cross_attn_grouped_kernel<G> (beam search) against float64."""
    from manual_whisper_b200 import _lib
    d = heads * 64
    worst = 0.0
    for T in CROSS_T:
        for B in (1, 3):
            g = torch.Generator(device=DEV).manual_seed(T * 10 + B + heads)
            per_unr = {}
            for G, unr in CROSS_G:
                q, kv = _cross_inputs(mode, B, G, T, heads, g) if unr != 8 else per_unr["inputs"]
                if unr == 4:
                    per_unr["inputs"] = (q, kv)
                out = torch.full((B * G + 1, d), float("nan"), device=DEV, dtype=_h16())
                _lib.check(lib.mw_step_cross_attention_h16(_ptr(q), _ptr(kv), B, G, T, heads, unr, _ptr(out), _stream()),
                           "mw_step_cross_attention_h16")
                torch.cuda.synchronize()
                assert torch.isnan(out[B * G:].float()).all()
                got = out[:B * G].view(B, G, heads, 64)
                k = kv[:, :d].view(B, 1, T, heads, 64).permute(0, 1, 3, 2, 4)      # [B, 1, heads, T, 64]
                v = kv[:, d:].view(B, 1, T, heads, 64).permute(0, 1, 3, 2, 4)
                ref, bound = _attend(q.view(B, G, heads, 64), k, v)
                worst = max(worst, _check_bound(got, ref, bound, f"cross {mode} T={T} B={B} G={G} unr={unr}"))
                if G == 1:
                    per_unr[unr] = out[:B * G]
            assert torch.equal(per_unr[4], per_unr[8]), f"T={T} B={B}: unr 4 and unr 8 differ"
    _report(f"cross-attention {mode} heads={heads}", worst)


def test_cross_attention_score_buffer_over_budget_is_an_error(lib):
    """The grouped kernel keeps G*T fp32 scores in shared memory (96 KB): beyond that the call fails before launching."""
    heads, d, G, B = 6, 384, 8, 1
    T = 96 * 1024 // (4 * G) + 1
    q = torch.zeros(B * G, d, device=DEV, dtype=_h16())
    kv = torch.zeros(B * T, 2 * d, device=DEV, dtype=_h16())
    out = torch.full((B * G, d), float("nan"), device=DEV, dtype=_h16())
    assert lib.mw_step_cross_attention_h16(_ptr(q), _ptr(kv), B, G, T, heads, 0, _ptr(out), _stream()) == 1
    assert b"shared memory" in lib.mw_last_error()
    torch.cuda.synchronize()
    assert torch.isnan(out.float()).all()
    # one key fewer fits
    assert lib.mw_step_cross_attention_h16(_ptr(q), _ptr(kv), B, G, T - 1, heads, 0, _ptr(out), _stream()) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
