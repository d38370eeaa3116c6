"""The encoder-side tensor-core kernels pinned against float64 references in every geometry their callers use: the
persistent tcgen05 GEMM (csrc/gemm.cu), the tcgen05 flash attention (csrc/attention.cu) and the LayerNorm variants
(csrc/elementwise.cu), through mw_gemm_general_h16, mw_attention_general_h16 and mw_layernorm_mode (include/mw_b200.h).

The conventions are those of tests/test_gpu_decode_step.py: references in float64 on the device from the exact 16-bit
inputs, every element held to a bound scaled to THAT element, NaN sentinels wherever a kernel must not write, bit-for-bit
asserts for every same-bits claim of the code, and the worst |err| / bound printed per case.

  * GEMM: 2^-18 sqrt(K) (|A| |W|^T) + 2^-22 (|bias| + |pre|), x 1.2 through GELU, + 2^-22 (|resid| + |ref|), plus half an
    ulp + 2^-25 for 16-bit output (the projection bound of the decode-step file).  The epilogue's GELU uses the
    Abramowitz & Stegun 7.1.26 erf (|error| < 1.5e-7), and 1 + erf cancels for negative inputs: a float32 emulation of the
    epilogue errs by up to 2.6e-7 at v in [-4, -2], which 1.2 * 2^-22 |pre| (>= 5.7e-7 there) covers.
  * attention: with p_j = exp(s_j - max s) and l = sum_j p_j (float64),
        half-ulp(|ref|) + u_P sum_j p_j |v_j| / l + n_keys 2^-25 max|v| / l (fp16 only) + 2^-20 slack max|v| + 2^-25.
    The kernel rounds its un-normalised P (<= 2^8 times p_j) to 16 bits before P V but sums l in fp32, so every p_j
    carries a relative error u_P (2^-11 for fp16, 2^-8 for bf16).  An fp16 P below 2^-14 is subnormal and rounds with an
    absolute error of up to 2^-25 in the kernel's units, which are >= the reference's: n_keys 2^-25 max|v| / l bounds them
    all.  Scores are fp32 sums of 64 products: an error e in every score moves the output by up to 2 e max|v|, and
    2^-20 slack max|v| (slack = max_j sum_i |q_i k_ij| / 8, _score_slack_rows) is 4x that.  The lazy rescale's exponent
    arithmetic errs by 2^-24 |max s| log2(e) / 8 in log2 units, below the same term.
  * LayerNorm: half-ulp(|y|) + 2^-18 (|gamma| + 1) + 2^-25 (the bound of test_layernorm_projection), x 1.2 through GELU,
    plus 2^-21 |y| for the f32 GELU (erff is accurate to a few ulp); the f32 outputs drop the half ulp.
"""
import pytest
import torch

from test_gpu_decode_step import _check_bound, _h16, _half_ulp, _layernorm_ref, _ptr, _report, _stream

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
NAN = float("nan")


@pytest.fixture(scope="module")
def lib():
    from manual_whisper_b200 import _lib
    return _lib.load()


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


# ================================================================================================ GEMM
class GemmCase:
    """One GemmArgs geometry (csrc/gemm.cuh) with seeded inputs.  resid: None, "separate" ([rows, ldr] f32, rows of batch b
    start at b * rbr), "broadcast" (rbr = 0: the positional embedding of conv2) or "inplace" (resid == out, f32)."""

    def __init__(self, what, *, M, N, K, batch=1, ars=None, abs_=0, a_off=0, a_len=None, bias=True, gelu=False, f32=False,
                 resid=None, rbr=0, ldr=None, obr=0, off=0, ldo=None, out_rows=None, out_col=0, seed=0):
        self.what, self.M, self.N, self.K, self.batch = what, M, N, K, batch
        self.ars = K if ars is None else ars
        self.abs_, self.a_off, self.gelu, self.f32, self.resid = abs_, a_off, gelu, f32, resid
        self.obr, self.off, self.out_col = obr, off, out_col
        self.ldo = N if ldo is None else ldo
        self.out_rows = (batch - 1) * obr + off + M if out_rows is None else out_rows
        if a_len is None:
            a_len = a_off + (batch - 1) * abs_ + (M - 1) * self.ars + K
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.a = (torch.randn(a_len, device=DEV, generator=g) * 0.5).to(_h16())
        self.w = (torch.randn(N, K, device=DEV, generator=g) * 0.05).to(_h16())
        self.bias = torch.randn(N, device=DEV, generator=g) * 0.1 if bias else None
        self.out_dtype = torch.float32 if f32 else _h16()
        self.rbr, self.ldr, self.res = rbr, N if ldr is None else ldr, None
        if resid == "inplace":
            assert f32 and off == 0
            self.rbr, self.ldr = obr, self.ldo
            self.out_init = torch.randn(self.out_rows, self.ldo, device=DEV, generator=g)
        else:
            self.out_init = torch.full((self.out_rows, self.ldo), NAN, device=DEV, dtype=self.out_dtype)
            if resid == "separate":
                self.res = torch.randn((batch - 1) * rbr + M, self.ldr, device=DEV, generator=g)
            elif resid == "broadcast":
                self.rbr = 0
                self.res = torch.randn(M, self.ldr, device=DEV, generator=g)

    def launch(self, lib, out, *, batch=None, b0=0, M=None, a=None, a_strides=None, resid_buf=None):
        """One call on out (a clone of out_init) for batch items b0 .. b0 + batch; a / a_strides replace A and its strides."""
        batch = self.batch if batch is None else batch
        M = self.M if M is None else M
        if a is None:
            ars, abs_ = self.ars, self.abs_
            a_ptr = self.a.data_ptr() + (self.a_off + b0 * abs_) * 2
        else:
            ars, abs_ = a_strides
            a_ptr = a.data_ptr() + b0 * abs_ * 2
        es = out.element_size()
        out_ptr = out.data_ptr() + (b0 * self.obr * self.ldo + self.out_col) * es
        if self.resid is None:
            r_ptr = None
        elif self.resid == "inplace":
            r_ptr = out_ptr if resid_buf is None else resid_buf.data_ptr() + (b0 * self.obr * self.ldo + self.out_col) * 4
        else:
            r_ptr = self.res.data_ptr() + b0 * self.rbr * self.ldr * 4
        from manual_whisper_b200 import _lib
        _lib.check(lib.mw_gemm_general_h16(a_ptr, ars, abs_, _ptr(self.w), self.K, _ptr(self.bias), r_ptr, self.rbr, self.ldr,
                                           out_ptr, self.obr, self.off, self.ldo, batch, M, self.N, self.K, int(self.gelu),
                                           int(self.f32), _stream()), f"mw_gemm_general_h16 {self.what}")
        torch.cuda.synchronize()
        return out

    def rows(self, batch=None, b0=0):
        batch = self.batch if batch is None else batch
        b = torch.arange(b0, b0 + batch, device=DEV)
        return (b[:, None] * self.obr + self.off + torch.arange(self.M, device=DEV)[None]).reshape(-1)

    def region(self, out, batch=None, b0=0):
        batch = self.batch if batch is None else batch
        return out[self.rows(batch, b0)][:, self.out_col:self.out_col + self.N].reshape(batch, self.M, self.N)

    def a_view(self):
        return torch.as_strided(self.a, (self.batch, self.M, self.K), (self.abs_, self.ars, 1), self.a_off)

    def reference(self):
        ad, wd = self.a_view().double(), self.w.double()
        pre = ad @ wd.t()
        mag = ad.abs() @ wd.abs().t()
        bound = 2.0 ** -18 * self.K ** 0.5 * mag
        if self.bias is not None:
            pre = pre + self.bias.double()
            bound = bound + 2.0 ** -22 * self.bias.double().abs()
        bound = bound + 2.0 ** -22 * pre.abs()
        ref = pre
        if self.gelu:
            ref = 0.5 * pre * (1.0 + torch.erf(pre / 2.0 ** 0.5))
            bound = bound * 1.2
        if self.resid is not None:
            if self.resid == "inplace":
                r = self.region(self.out_init).double()
            else:
                r = torch.as_strided(self.res, (self.batch, self.M, self.N), (self.rbr * self.ldr, self.ldr, 1)).double()
            ref = ref + r
            bound = bound + 2.0 ** -22 * r.abs()
        bound = bound + 2.0 ** -22 * ref.abs()
        if not self.f32:
            bound = bound + _half_ulp() * ref.abs() + 2.0 ** -25
        return ref, bound


def _run_gemm_case(lib, c):
    """Bound check plus the same-bits claims: two runs, each batch item == its batch-1 run, the overlapping-row map == a
    materialised im2col copy, in-place residual == out-of-place.  Everything outside the output region keeps its bits."""
    out = c.launch(lib, c.out_init.clone())
    ref, bound = c.reference()
    worst = _check_bound(c.region(out), ref, bound, c.what)
    outside = torch.ones(out.shape, dtype=torch.bool, device=DEV)
    outside[c.rows()[:, None], torch.arange(c.out_col, c.out_col + c.N, device=DEV)[None]] = False
    assert torch.equal(_bits(out)[outside], _bits(c.out_init)[outside]), f"{c.what}: wrote outside its output region"
    assert _same_bits(c.launch(lib, c.out_init.clone()), out), f"{c.what}: two runs differ"
    if c.batch > 1:
        for b in range(c.batch):
            one = c.launch(lib, c.out_init.clone(), batch=1, b0=b)
            assert _same_bits(c.region(one, 1, b), c.region(out, 1, b)), f"{c.what}: batch item {b} != its batch-1 run"
    if c.ars != c.K:
        im2col = c.a_view().contiguous()
        mat = c.launch(lib, c.out_init.clone(), a=im2col, a_strides=(c.K, c.M * c.K))
        assert _same_bits(c.region(mat), c.region(out)), f"{c.what}: overlapping rows != materialised im2col"
    if c.resid == "inplace":
        sep = c.launch(lib, torch.full_like(c.out_init, NAN), resid_buf=c.out_init.clone())
        assert _same_bits(c.region(sep), c.region(out)), f"{c.what}: in-place residual != out-of-place"
    return worst


# (n_mels, d_model, ffn, n_audio_ctx) of the encoder-side shapes: tiny, small, large-v3 and the test-small dims
ENC = {"tiny": (80, 384, 1536, 1500), "small": (80, 768, 3072, 1500), "large-v3": (128, 1280, 5120, 1500),
       "test-small": (80, 128, 512, 200)}
SITES = ["conv1", "conv2", "qkv", "out", "fc1", "fc2", "cross_kv", "prefill"]


def _model_cases(model, site, B):
    n, d, ffn, T = ENC[model]
    F = 2 * T
    s = 1000 * list(ENC).index(model) + 100 * SITES.index(site) + B
    if site == "conv1":       # time-major features [B, F+2, n_mels]; h1 rows 0 and F+1 of every item are NaN sentinels
        return [GemmCase(f"{model} conv1 B={B}", batch=B, M=F, N=d, K=3 * n, ars=n, abs_=(F + 2) * n, a_len=B * (F + 2) * n,
                         gelu=True, obr=F + 2, off=1, out_rows=B * (F + 2), seed=s)]
    if site == "conv2":       # stride-2 rows of h1, positional embedding broadcast over the batch
        return [GemmCase(f"{model} conv2 B={B}", batch=B, M=T, N=d, K=3 * d, ars=2 * d, abs_=(F + 2) * d,
                         a_len=B * (F + 2) * d, gelu=True, f32=True, resid="broadcast", obr=T, seed=s)]
    M = B * T
    if site == "qkv":
        return [GemmCase(f"{model} qkv B={B}", M=M, N=3 * d, K=d, seed=s)]
    if site == "out":
        return [GemmCase(f"{model} out-proj B={B}", M=M, N=d, K=d, f32=True, resid="inplace", seed=s)]
    if site == "fc1":
        return [GemmCase(f"{model} fc1 B={B}", M=M, N=ffn, K=d, gelu=True, seed=s)]
    if site == "fc2":
        return [GemmCase(f"{model} fc2 B={B}", M=M, N=d, K=ffn, f32=True, resid="inplace", seed=s)]
    if site == "cross_kv":
        return [GemmCase(f"{model} cross K/V B={B}", M=M, N=2 * d, K=d, seed=s)]
    cases = []                # the six projections of the batched prompt prefill
    for Pm in (5, 28, 223):
        M = B * Pm
        cases += [GemmCase(f"{model} prefill qkv B={B} Pm={Pm}", M=M, N=3 * d, K=d, seed=s + Pm),
                  GemmCase(f"{model} prefill out B={B} Pm={Pm}", M=M, N=d, K=d, f32=True, resid="inplace", seed=s + Pm + 1),
                  GemmCase(f"{model} prefill cross q B={B} Pm={Pm}", M=M, N=d, K=d, seed=s + Pm + 2),
                  GemmCase(f"{model} prefill cross out B={B} Pm={Pm}", M=M, N=d, K=d, f32=True, resid="inplace", seed=s + Pm + 3),
                  GemmCase(f"{model} prefill fc1 B={B} Pm={Pm}", M=M, N=ffn, K=d, gelu=True, seed=s + Pm + 4),
                  GemmCase(f"{model} prefill fc2 B={B} Pm={Pm}", M=M, N=d, K=ffn, f32=True, resid="inplace", seed=s + Pm + 5)]
    return cases


@pytest.mark.parametrize("site", SITES)
@pytest.mark.parametrize("model", list(ENC))
def test_gemm_model_sites(lib, model, site):
    """The encoder's conv stem (implicit GEMM on overlapping rows), its layer projections, the cross K/V projection and the
    prefill projections, each at B = 1 and 3, in the geometry model.cu / decoder.cu launch them."""
    worst = 0.0
    for B in (1, 3):
        for c in _model_cases(model, site, B):
            worst = max(worst, _run_gemm_case(lib, c))
    _report(f"gemm {model} {site}", worst)


# wav2vec2 (csrc/w2v.cu): feature-extractor convs, kernel k, stride 2, over C channels
W2V_CONVS = [(C_, k, form) for C_ in (512, 128) for k in (3, 2) for form in ("xlsr", "base", "base_last")]


@pytest.mark.parametrize("C_,k,form", W2V_CONVS, ids=[f"C{c}-k{k}-{f}" for c, k, f in W2V_CONVS])
def test_gemm_w2v_conv(lib, C_, k, form):
    """Row stride 2C, K = kC, batch stride T_{l-1} C with T_{l-1} odd and even.  XLSR form: bias, f32 (a LayerNorm follows);
    base form: GELU, 16-bit, the last layer f32."""
    worst = 0.0
    for T_prev in ((1999, 2000) if C_ == 512 else (399, 400)):
        M = (T_prev - k) // 2 + 1
        for n in (1, 3):
            xlsr = form == "xlsr"
            c = GemmCase(f"w2v conv C={C_} k={k} {form} T_prev={T_prev} n={n}", batch=n, M=M, N=C_, K=k * C_, ars=2 * C_,
                         abs_=T_prev * C_, a_len=n * T_prev * C_, bias=xlsr, gelu=not xlsr, f32=form != "base", obr=M,
                         seed=T_prev + n + k)
            worst = max(worst, _run_gemm_case(lib, c))
    _report(f"gemm w2v conv C={C_} k={k} {form}", worst)


# positional conv: (d, groups, kernel); d / groups = 64 adds in place into x, 48 writes 64 padded columns into a scratch buffer
W2V_POS = [(1024, 16, 128), (128, 2, 16), (768, 16, 128)]


@pytest.mark.parametrize("d,G,kp", W2V_POS, ids=[f"d{d}-G{G}-kp{kp}" for d, G, kp in W2V_POS])
def test_gemm_w2v_pos_conv(lib, d, G, kp):
    """One implicit GEMM per group over the group-major copy xg [n, G, T + kp, gw]: row stride gw, K = kp gw, N = 64.
    gw = 64: x[:, 64g : 64g + 64] += GELU(conv + bias) in place (res_batch_rows = T); every other group's columns keep their
    bits.  gw = 48: columns 64g .. 64g + 64 of the scratch [n T, 64 G]; the other columns stay NaN."""
    gw = d // G
    worst = 0.0
    for T in (1499, 249):
        for n in (1, 3):
            for grp in sorted({0, G - 1}):
                kw = dict(batch=n, M=T, N=64, K=kp * gw, ars=gw, abs_=G * (T + kp) * gw, a_off=grp * (T + kp) * gw,
                          a_len=n * G * (T + kp) * gw, f32=True, obr=T, out_rows=n * T, out_col=64 * grp, seed=T + n + grp)
                what = f"w2v pos conv d={d} G={G} kp={kp} T={T} n={n} g={grp}"
                if gw == 64:
                    c = GemmCase(what, gelu=True, resid="inplace", ldo=d, **kw)
                else:
                    c = GemmCase(what, bias=False, ldo=64 * G, **kw)
                worst = max(worst, _run_gemm_case(lib, c))
    _report(f"gemm w2v pos conv d={d} G={G} kp={kp}", worst)


@pytest.mark.parametrize("C_,d,vocab", [(512, 1024, 3503), (128, 128, 32)])
def test_gemm_w2v_heads(lib, C_, d, vocab):
    """The feature projection (K = C) and the lm_head (N = vocab padded to 32: 3520 > 1024 with N % 256 != 0, or 32)."""
    worst = 0.0
    for n in (1, 3):
        M = n * 1499
        N = (vocab + 31) // 32 * 32
        worst = max(worst, _run_gemm_case(lib, GemmCase(f"w2v feature projection C={C_} n={n}", M=M, N=d, K=C_, f32=True, seed=n)))
        worst = max(worst, _run_gemm_case(lib, GemmCase(f"w2v lm_head vocab={vocab} n={n}", M=M, N=N, K=d, f32=True, seed=n + 7)))
    _report(f"gemm w2v heads C={C_} d={d} vocab={vocab}", worst)


def check_gemm_contiguous(lib, M, N, K, mode):
    """A contiguous product against float64 (mode plain, bias_gelu or bias_resid_f32); the first M rows of a 2M-row call equal
    the M-row call bit for bit.  Also the body of tests/test_gpu_kernels.py::test_gemm."""
    kw = dict(bias=mode != "plain", gelu=mode == "bias_gelu", f32=mode == "bias_resid_f32",
              resid="separate" if mode == "bias_resid_f32" else None, seed=M * 7 + N)
    worst = _run_gemm_case(lib, GemmCase(f"gemm {M}x{N}x{K} {mode}", M=M, N=N, K=K, **kw))
    two = GemmCase(f"gemm {2 * M}x{N}x{K} {mode}", M=2 * M, N=N, K=K, **kw)
    full = two.launch(lib, two.out_init.clone())
    half = two.launch(lib, two.out_init.clone(), M=M)
    assert _same_bits(half[:M], full[:M]), "the first M rows of a 2M-row call differ from the M-row call"
    assert torch.isnan(half[M:].float()).all(), "the M-row call wrote past row M"
    _report(f"gemm {M}x{N}x{K} {mode}", worst)


# the M tile edges, K below one 16-wide MMA and below one 64-wide K block, N of one 32-column chunk and N = 1056 (> 1024:
# 256-wide tiles, the last one 32 wide); tests/test_gpu_kernels.py::test_gemm runs the same checks on nine more shapes, among
# them (4096, 5120, 1280): 640 tiles, more than two per SM
EDGE_SHAPES = [(M, 32, 8) for M in (1, 127, 128, 129)] + [(M, 1056, 56) for M in (1, 127, 128, 129)]


@pytest.mark.parametrize("mode", ["plain", "bias_gelu", "bias_resid_f32"])
@pytest.mark.parametrize("M,N,K", EDGE_SHAPES)
def test_gemm_edges(lib, M, N, K, mode):
    """Contiguous products at the tile edges."""
    check_gemm_contiguous(lib, M, N, K, mode)


# ================================================================================================ attention
MODES = ["random", "rise", "maxkey", "lowall", "huge", "subnormal"]
PAD = 6.0e4


def _qkv_inputs(B, Tq, Tk, H, mode, lens, seed):
    """q [B, Tq, H, 64], k, v [B, Tk, H, 64] (16-bit) with the score pattern of `mode` over the valid keys (lens[b]):
      rise:      one row in every 32 (rows 7 mod 32) has a block maximum 60 raw units (> 44.4 = 2^8 in the exponent) above
                 the previous block's in every key block: its warp rescales O at every j > 0, decided by that row alone;
      maxkey:    rows 3 mod 8 peak only at key 0, rows 5 mod 8 only at the last valid key (in a partial block when T % 64 != 0);
      lowall:    every valid score <= -100, so a masked key that leaked (score ~0) would dominate;
      huge:      scores of magnitude ~1000;
      subnormal: an early spike with every other key 14-24 log2 units below it (fp16-subnormal P)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    q = torch.randn(B, Tq, H, 64, device=DEV, generator=g)
    k = torch.randn(B, Tk, H, 64, device=DEV, generator=g)
    v = torch.randn(B, Tk, H, 64, device=DEV, generator=g)
    rows = torch.arange(Tq, device=DEV)
    keys = torch.arange(Tk, device=DEV)
    if mode == "rise":
        sel = rows % 32 == 7
        q[:, :, :, 0] = 0.0
        q[:, sel] = 0.0
        q[:, sel, :, 0] = 8.0
        k[:, :, :, 0] = (7.5 * (keys // 64) + 0.03125 * (keys % 64))[None, :, None]
    elif mode == "maxkey":
        q[:, :, :, 1:3] = 0.0
        q[:, rows % 8 == 3, :, 1] = 8.0
        q[:, rows % 8 == 5, :, 2] = 8.0
        k[:, :, :, 1:3] = 0.0
        k[:, 0, :, 1] = 8.0
        for b in range(B):
            k[b, lens[b] - 1, :, 2] = 8.0
    elif mode == "lowall":
        q[:, :, :, 0] = 8.0
        k[:, :, :, 0] = -20.0
    elif mode == "huge":
        q, k = q * 11.2, k * 11.2
    elif mode == "subnormal":
        q = q * 0.25
        q[:, :, :, 3] = 8.0
        k[:, :, :, 3] = 3.5 + 6.7 * torch.rand(B, Tk, H, device=DEV, generator=g)
        k[:, min(1, Tk - 1), :, 3] = 20.0
    return q.to(_h16()), k, v


def _score_slack_rows(q, k):
    """max_j sum_i |q_i k_ij| / 8 per query row: q [..., Tq, 64], k [..., n, 64] -> [..., Tq]"""
    return (q.double().abs() @ k.double().abs().transpose(-1, -2)).amax(-1) / 8.0


def _attention_ref(q, k, v):
    """float64 attention of q [..., Tq, 64] over k, v [..., n, 64] (16-bit values) and the bound of the module docstring."""
    qd, kd, vd = q.double(), k.double(), v.double()
    s = qd @ kd.transpose(-1, -2) / 8.0
    p = torch.exp(s - s.amax(-1, keepdim=True))
    l = p.sum(-1, keepdim=True)
    ref = (p @ vd) / l
    vmax = vd.abs().amax(-2, keepdim=True)
    bound = _half_ulp() * ref.abs() + _half_ulp() * (p @ vd.abs()) / l + 2.0 ** -20 * _score_slack_rows(q, k).unsqueeze(-1) * vmax
    if _h16() == torch.float16:
        bound = bound + k.shape[-2] * 2.0 ** -25 * vmax / l
    return ref, bound + 2.0 ** -25


def _attn_general(lib, q, ldq, colq0, kv, ldkv, colk0, colv0, out, out_ld, B, Tq, Tk, H, lens=None):
    from manual_whisper_b200 import _lib
    _lib.check(lib.mw_attention_general_h16(_ptr(q), ldq, colq0, _ptr(kv), ldkv, colk0, colv0, _ptr(out), out_ld, B, Tq, Tk, H,
                                            _ptr(lens), _stream()), "mw_attention_general_h16")
    torch.cuda.synchronize()
    return out


def _heads(x):
    """[B, T, H, 64] -> [B, H, T, 64]"""
    return x.permute(0, 2, 1, 3)


def check_self_attention(lib, B, T, H, mode):
    """The encoder's self-attention (mw_attention_h16 on packed q|k|v) against float64; the general form on separate q and
    k|v buffers at other column offsets gives the same bits.  Also the body of tests/test_gpu_kernels.py::
    test_encoder_attention."""
    from manual_whisper_b200 import _lib
    d = 64 * H
    q, k, v = _qkv_inputs(B, T, T, H, mode, [T] * B, seed=B * 7919 + T * 31 + H + MODES.index(mode))
    k16, v16 = k.to(_h16()), v.to(_h16())
    qkv = torch.cat([q.reshape(B * T, d), k16.reshape(B * T, d), v16.reshape(B * T, d)], dim=1).contiguous()
    out = torch.full((B * T + 1, d), NAN, device=DEV, dtype=_h16())
    _lib.check(lib.mw_attention_h16(_ptr(qkv), _ptr(out), B, T, H, _stream()), "mw_attention_h16")
    torch.cuda.synchronize()
    assert torch.isnan(out[B * T:].float()).all(), "wrote past the last row"
    ref, bound = _attention_ref(_heads(q), _heads(k16), _heads(v16))
    worst = _check_bound(_heads(out[:B * T].view(B, T, H, 64)), ref, bound, f"self-attention B={B} T={T} H={H} {mode}")
    # general form: q at column 64 of [B, T, d + 64], k | v at columns 64 / 64 + d of [B, T, 2d + 64], out_ld = d + 64
    qb = torch.randn(B, T, d + 64, device=DEV).to(_h16())
    qb[:, :, 64:] = q.reshape(B, T, d)
    kvb = torch.randn(B, T, 2 * d + 64, device=DEV).to(_h16())
    kvb[:, :, 64:64 + d] = k16.reshape(B, T, d)
    kvb[:, :, 64 + d:] = v16.reshape(B, T, d)
    gen = torch.full((B * T + 1, d + 64), NAN, device=DEV, dtype=_h16())
    _attn_general(lib, qb, d + 64, 64, kvb, 2 * d + 64, 64, 64 + d, gen, d + 64, B, T, T, H)
    assert _same_bits(gen[:B * T, :d], out[:B * T]), "general form on split buffers != packed qkv"
    assert torch.isnan(gen[:, d:].float()).all() and torch.isnan(gen[B * T:].float()).all(), "general form wrote outside its output"
    again = torch.full_like(out, NAN)
    _lib.check(lib.mw_attention_h16(_ptr(qkv), _ptr(again), B, T, H, _stream()), "mw_attention_h16")
    torch.cuda.synchronize()
    assert _same_bits(again, out), "two runs differ"
    _report(f"self-attention B={B} T={T} H={H} {mode}", worst)


# tile edges of T; tests/test_gpu_kernels.py::test_encoder_attention runs the same checks at (1, 1500, 20), (3, 1500, 6),
# (1, 200, 2), (1, 128, 1) and (2, 77, 4)
SELF_SHAPES = [(2, 1500, 6), (3, 200, 2), (1, 1, 1), (1, 63, 1), (1, 64, 2), (1, 65, 2), (2, 127, 4), (1, 129, 1)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B,T,H", SELF_SHAPES)
def test_self_attention(lib, B, T, H, mode):
    check_self_attention(lib, B, T, H, mode)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("H,Tk", [(6, 200), (6, 1500), (20, 200), (20, 1500)])
def test_cross_attention_general(lib, H, Tk, mode):
    """The batched prefill's cross-attention (decoder.cu: batched_prefill): Tq prompt rows per sequence over its Tk encoder
    rows, q [B, Tq, d] and k|v [B, Tk, 2d] in separate buffers."""
    d = 64 * H
    worst = 0.0
    for Tq in (4, 31, 128, 129, 223):
        for B in (1, 3):
            q, k, v = _qkv_inputs(B, Tq, Tk, H, mode, [Tk] * B, seed=Tq * 101 + B * 13 + Tk + H + MODES.index(mode))
            k16, v16 = k.to(_h16()), v.to(_h16())
            kv = torch.cat([k16.reshape(B * Tk, d), v16.reshape(B * Tk, d)], dim=1).contiguous()
            qc = q.reshape(B * Tq, d).contiguous()
            out = _attn_general(lib, qc, d, 0, kv, 2 * d, 0, d, torch.full((B * Tq + 1, d), NAN, device=DEV, dtype=_h16()), d,
                                B, Tq, Tk, H)
            assert torch.isnan(out[B * Tq:].float()).all(), "wrote past the last row"
            ref, bound = _attention_ref(_heads(q), _heads(k16), _heads(v16))
            what = f"cross-attention B={B} Tq={Tq} Tk={Tk} H={H} {mode}"
            worst = max(worst, _check_bound(_heads(out[:B * Tq].view(B, Tq, H, 64)), ref, bound, what))
            again = _attn_general(lib, qc, d, 0, kv, 2 * d, 0, d, torch.full_like(out, NAN), d, B, Tq, Tk, H)
            assert _same_bits(again, out), f"{what}: two runs differ"
    _report(f"cross-attention H={H} Tk={Tk} {mode}", worst)


RAGGED = [(T, d, H) for T in (1499, 249) for d, H in ((1024, 16), (768, 12), (128, 2))]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("T,d,H", RAGGED)
def test_ragged_attention(lib, T, d, H, mode):
    """The aligner's ragged self-attention (kv_lens): windows of lengths T, 1, 63, 64, 65, 200, T - 1 in one call.  The k and v
    parts of padded rows hold +-6e4; their q parts are ordinary.  Keys >= len must be masked; query rows of the tile holding the
    window's last row are written (padded rows: their attention over the valid keys), rows of wholly padded 128-row tiles keep
    their NaN sentinels.  With random scores each window equals its solo run (B = 1, T = len) bit for bit, the claim of
    mw_w2v_emissions; the score patterns can move a boundary warp's exponent reference through a padded row (kernels.cuh)."""
    from manual_whisper_b200 import _lib
    lens = [T, 1, 63, 64, 65, 200, T - 1]
    B = len(lens)
    q, k, v = _qkv_inputs(B, T, T, H, mode, lens, seed=T * 3 + d + MODES.index(mode))
    g = torch.Generator(device=DEV).manual_seed(T + d)
    for b, L in enumerate(lens):
        sign = torch.randint(0, 2, (2, T - L, H, 64), device=DEV, generator=g).float() * 2 - 1
        k[b, L:] = PAD * sign[0]
        v[b, L:] = PAD * sign[1]
    k16, v16 = k.to(_h16()), v.to(_h16())
    qkv = torch.cat([q.reshape(B * T, d), k16.reshape(B * T, d), v16.reshape(B * T, d)], dim=1).contiguous()
    lens_t = torch.tensor(lens, dtype=torch.int32, device=DEV)
    out = _attn_general(lib, qkv, 3 * d, 0, qkv, 3 * d, d, 2 * d, torch.full((B * T, d), NAN, device=DEV, dtype=_h16()), d, B, T,
                        T, H, lens_t)
    outv = out.view(B, T, H, 64)
    worst = 0.0
    for b, L in enumerate(lens):
        written = min(T, -(-L // 128) * 128)
        what = f"ragged T={T} d={d} {mode} window {b} len={L}"
        assert torch.isnan(outv[b, written:].float()).all(), f"{what}: a wholly padded query tile was written"
        ref, bound = _attention_ref(_heads(q[b:b + 1, :written]), _heads(k16[b:b + 1, :L]), _heads(v16[b:b + 1, :L]))
        worst = max(worst, _check_bound(_heads(outv[b:b + 1, :written]), ref, bound, what))
        if mode == "random":
            solo_qkv = qkv.view(B, T, 3 * d)[b, :L].contiguous()
            solo = _attn_general(lib, solo_qkv, 3 * d, 0, solo_qkv, 3 * d, d, 2 * d,
                                 torch.full((L, d), NAN, device=DEV, dtype=_h16()), d, 1, L, L, H)
            assert _same_bits(out.view(B, T, d)[b, :L], solo), f"{what}: differs from its solo run"
    again = _attn_general(lib, qkv, 3 * d, 0, qkv, 3 * d, d, 2 * d, torch.full_like(out, NAN), d, B, T, T, H, lens_t)
    assert _same_bits(again, out), "two runs differ"
    _report(f"ragged attention T={T} d={d} H={H} {mode}", worst)


# ================================================================================================ LayerNorm variants
def _ln_inputs(rows, d, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(rows, d, device=DEV, generator=g) * 3 + 1
    gam, bet = torch.randn(d, device=DEV, generator=g), torch.randn(d, device=DEV, generator=g)
    return x, gam, bet


def _ln_bound(y, gam, h16, gelu=False):
    b = 2.0 ** -18 * (gam.double().abs() + 1)
    if gelu:
        b = b * 1.2 + 2.0 ** -21 * y.abs()
    if h16:
        b = b + _half_ulp() * y.abs() + 2.0 ** -25
    return b + 2.0 ** -25


def _ln_call(lib, x, gam, bet, out, mode):
    from manual_whisper_b200 import _lib
    _lib.check(lib.mw_layernorm_mode(_ptr(x), _ptr(gam), _ptr(bet), _ptr(out), x.shape[0], x.shape[1], mode, _stream()),
               f"mw_layernorm_mode {mode}")
    torch.cuda.synchronize()
    return out


def check_layernorm(lib, rows, d):
    """mw_layernorm (mode 0): LN -> 16-bit against float64; mw_layernorm_mode 0 is the same launch.  The body of
    tests/test_gpu_kernels.py::test_layernorm."""
    from manual_whisper_b200 import _lib
    x, gam, bet = _ln_inputs(rows, d, d)
    out = torch.full((rows + 1, d), NAN, device=DEV, dtype=_h16())
    _lib.check(lib.mw_layernorm(_ptr(x), _ptr(gam), _ptr(bet), _ptr(out), rows, d, _stream()), "mw_layernorm")
    torch.cuda.synchronize()
    assert torch.isnan(out[rows:].float()).all()
    y = _layernorm_ref(x, gam, bet)
    worst = _check_bound(out[:rows], y, _ln_bound(y, gam, True), f"layernorm rows={rows} d={d}")
    assert _same_bits(_ln_call(lib, x, gam, bet, torch.full_like(out[:rows], NAN), 0), out[:rows])
    _report(f"layernorm rows={rows} d={d}", worst)


@pytest.mark.parametrize("rows,d", [(1, 128), (37, 128), (4097, 128), (1, 512), (999, 512), (2999, 512)])
def test_layernorm_gelu(lib, rows, d):
    """Modes 1 and 2 (the wav2vec2 feature extractor): GELU(LN) -> 16-bit and -> f32; mode 1 == mode 2 rounded to 16 bits."""
    x, gam, bet = _ln_inputs(rows, d, rows + d)
    y = _layernorm_ref(x, gam, bet)
    gy = 0.5 * y * (1.0 + torch.erf(y / 2.0 ** 0.5))
    hb = torch.full((rows + 1, d), NAN, device=DEV, dtype=_h16())
    h = _ln_call(lib, x, gam, bet, hb[:rows], 1)
    assert torch.isnan(hb[rows:].float()).all(), "wrote past the last row"
    f = _ln_call(lib, x, gam, bet, torch.full((rows, d), NAN, device=DEV), 2)
    worst = _check_bound(h, gy, _ln_bound(gy, gam, True, gelu=True), f"layernorm mode 1 rows={rows} d={d}")
    worst = max(worst, _check_bound(f, gy, _ln_bound(gy, gam, False, gelu=True), f"layernorm mode 2 rows={rows} d={d}"))
    assert _same_bits(h, f.to(_h16())), "mode 1 != mode 2 rounded to 16 bits"
    assert _same_bits(_ln_call(lib, x, gam, bet, torch.full_like(f, NAN), 2), f), "two runs differ"
    _report(f"layernorm GELU rows={rows} d={d}", worst)


@pytest.mark.parametrize("rows,d", [(1, 384), (37, 384), (2999, 384), (1, 768), (999, 768), (1, 1024), (37, 1024), (2999, 1024)])
def test_layernorm_dual(lib, rows, d):
    """Mode 3 (post-LayerNorm wav2vec2-base layers): LN written back over x in f32 plus a 16-bit copy; the copy equals
    mw_layernorm's output and the written-back f32 rounded to 16 bits."""
    from manual_whisper_b200 import _lib
    x, gam, bet = _ln_inputs(rows, d, rows * 3 + d)
    y = _layernorm_ref(x, gam, bet)
    plain = torch.full((rows, d), NAN, device=DEV, dtype=_h16())
    _lib.check(lib.mw_layernorm(_ptr(x), _ptr(gam), _ptr(bet), _ptr(plain), rows, d, _stream()), "mw_layernorm")
    xw = x.clone()
    h = _ln_call(lib, xw, gam, bet, torch.full((rows, d), NAN, device=DEV, dtype=_h16()), 3)
    worst = _check_bound(h, y, _ln_bound(y, gam, True), f"layernorm mode 3 h16 rows={rows} d={d}")
    worst = max(worst, _check_bound(xw, y, _ln_bound(y, gam, False), f"layernorm mode 3 f32 rows={rows} d={d}"))
    assert not torch.equal(xw, x), "mode 3 did not write x back"
    assert _same_bits(h, plain), "mode 3's 16-bit output != mw_layernorm's"
    assert _same_bits(h, xw.to(_h16())), "mode 3's 16-bit output != its written-back f32 rounded to 16 bits"
    _report(f"layernorm mode 3 rows={rows} d={d}", worst)
