"""Per-kernel parity of the forward sequence path on a real B200 (pytest -m gpu): the tcgen05 GEMM / conv with its fused
epilogue (gemm_tc.cuh, gemm_epilogue.cuh) and flash attention (attention_tc.cuh).  The GEMM is called through tts_k_gemm_epi,
which hands every GemmParams field to the launcher the library itself uses; each case takes its launch configuration from a
call site of the encoder, decoder, postnet, heads or training step and is named after it.  Attention is called through
tts_k_attention_strided with the strides of the library's own calls.

GEMM, exact mode.  A and W are integers with |v| <= 2, bias and residual are integers, pe is a multiple of 1/8 and alpha = 0.5:
the accumulator is an exact integer whatever the accumulation order, and alpha * pe is exact with or without an FMA.  The
reference is an fp64 GEMM followed by the epilogue in float32 torch ops in the kernel's order (bias, alpha * pe, word dropout
as ONE fp32 multiply by the same fp32 scale, residual, activation, bit dropout, length mask), dropout masks from
oracle/philox.py.  fp32 outputs must match bit for bit and bf16 outputs must equal bf16(reference) (both round to nearest
even).  tanh differs from torch's by a few fp32 ulp, so tanh sites allow one bf16 ulp after the rounding.
GEMM, random mode.  Gaussian operands; |err| <= 1e-4 * (the same computation on |A| |W| |bias| |alpha pe| |resid|), plus one
bf16 ulp of the reference for bf16 outputs.
Both forms.  The epilogue exists twice: the 16-byte vector form (with the TMA store) and the scalar gemm_store, which takes
the scatters, columns past the last full 32-column chunk and any layout the vector form cannot address.  Every plain-matrix
case runs a second time with ldo (and ldr) off a multiple of 8, which forces the scalar form, and both results must be
bit-identical.  Every output buffer starts as a NaN sentinel; columns past N, rows past M and the padding of ldo must keep it.

Attention.  Against an fp64 softmax of the same bf16 inputs.  The kernel rounds each probability p to bf16 for the P.V
product (relative error <= 2^-8, the unit roundoff of an 8-bit significand) while l = sum p stays fp32; every fourth pair of
exponentials comes from a polynomial with relative error 7.7e-5 (the others from ex2.approx, 2^-22); the scores carry the
fp32 accumulation error of Q.K (<= 64 * 2^-24 * sum |q||k|, times the log2 scale), and O accumulates Lk / 16 MMAs in fp32.
With c = 2^-8 + 2 * (7.7e-5 + e_s) + Lk * 2^-23 (c ~ 2.1 * 2^-9 for the production shapes) the bound per output is
    |O - O_ref| <= c * (sum_j p_j |v_j|) / (sum_j p_j) + ulp_bf16(O_ref)
where the last term is the final rounding of O to bf16.  lse (log2 domain, consumed by the backward pass) carries only the
errors of l: |lse - lse_ref| <= (7.7e-5 + e_s + Lk 2^-24) / ln 2 + 2^-22 |lse_ref|."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

F64 = torch.float64
F32_SENT = 0x7FC0DEAD                     # quiet NaN with a payload: never produced by the kernel
BF16_SENT = 0x7FDE
SEED = 0x0123_4567_89AB_CDEF              # both Philox key halves non-zero
SC_NONE, SC_CROSS_KV, SC_HEAD, SC_CROSS_KV_VT = 0, 1, 2, 3
P_WORD = 0.1
THRESH = int(P_WORD * 4294967296.0)
DSCALE = float(torch.tensor(1.0) / torch.tensor(1.0 - P_WORD))      # the fp32 scale the training step passes


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from transformer_tacotron2_b200 import _lib
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    return _lib.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _ints(shape, g, lo=-2, hi=2, dtype=torch.bfloat16):
    return torch.randint(lo, hi + 1, shape, generator=g, device="cuda").to(dtype)


def _bf16_ulp(x):
    a = x.abs().clamp(min=2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def _sentinel(shape, dtype):
    if dtype == torch.float32:
        return torch.full(shape, F32_SENT, dtype=torch.int32, device="cuda").view(torch.float32)
    return torch.full(shape, BF16_SENT, dtype=torch.int16, device="cuda").view(torch.bfloat16)


def _is_sentinel(t):
    if t.dtype == torch.float32:
        return bool((t.view(torch.int32) == F32_SENT).all())
    return bool((t.view(torch.int16) == BF16_SENT).all())


def _bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def _gemm_epi(lib, **kw):
    from transformer_tacotron2_b200 import _lib
    a = _lib.TtsKGemm()
    a.struct_size = C.sizeof(_lib.TtsKGemm)
    a.taps, a.drop_site, a.dropw_site, a.B = 1, -1, -1, 1
    for k, v in kw.items():
        setattr(a, k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
    return lib.tts_k_gemm_epi(C.byref(a), _stream())


# ================================================================================================ GEMM cases
# Launch configuration of each call site (tts_b200.cu: run_encoder, run_decoder_tf, run_postnet_rows; train.cuh: the training
# forward and the input-gradient GEMMs).  out: "bf16" / "f32" (ldo = N unless given); resid: "bf16" / "f32" (ldr = N unless
# given); pe: "alpha" / "alpha_ptr"; drop (bit dropout, p = 0.5): "seed" / "seed_ptr"; dropw: word-dropout site (p = 0.1).
SITES = {
    "enc_conv": dict(N=512, K=512, taps=5, act=1, lens=True, out="bf16"),
    "enc_proj": dict(N=512, K=512, pe="alpha", out="bf16"),
    "pre_proj": dict(N=512, K=256, pe="alpha_ptr", out="bf16"),
    "qkv": dict(N=1536, K=512, out="bf16"),
    "wo": dict(N=512, K=512, resid="bf16", out="f32"),
    "w1": dict(N=2048, K=512, act=1, out="bf16"),
    "w2": dict(N=512, K=2048, resid="bf16", out="f32"),
    "prenet_fc1": dict(N=256, K=96, act=1, drop="seed", out="bf16"),
    "prenet_fc1_seed_ptr": dict(N=256, K=96, act=1, drop="seed_ptr", out="bf16"),
    "prenet_fc2": dict(N=256, K=256, act=1, drop="seed_ptr", out="bf16"),
    "train_enc_proj": dict(N=512, K=512, pe="alpha_ptr", dropw=16, out="bf16"),
    "train_wo": dict(N=512, K=512, dropw=64, resid="bf16", out="f32"),
    "train_cross_kv": dict(N=6144, K=512, out="bf16"),
    "dgrad_resid": dict(N=512, K=1536, resid="f32", out="f32"),
    "post_conv0": dict(N=512, K=96, taps=5, act=2, lens=True, out="bf16"),
    # N = 80: chunks 0 and 1 take the vector form and the TMA store, chunk 2 (columns 64..79) the scalar form
    "post_conv4": dict(N=80, K=512, taps=5, resid="f32", lens=True, out="f32"),
    "head": dict(N=81, K=512, lens=True, scatter=SC_HEAD),
    # no call site combines all seven stages; these two pin their order (a residual added after the activation, say)
    "every_stage_bf16": dict(N=512, K=512, pe="alpha_ptr", dropw=64, resid="bf16", act=2, drop="seed_ptr", lens=True, out="bf16"),
    "every_stage_f32": dict(N=512, K=256, pe="alpha", dropw=17, resid="f32", act=1, drop="seed", lens=True, out="f32"),
}
# (T, lens): utterances of T rows, ragged lengths; 128-row tiles straddle utterances
TOKENS = {"T1": (1, [1, 0, 1]), "T37": (37, [37, 20, 1, 36]), "T129": (129, [129, 64, 65]), "T200": (200, [200, 1, 137])}
UTT_OFFSET = 5


def _make_inputs(c, T, lens, exact, seed):
    N, K, taps = c["N"], c["K"], c.get("taps", 1)
    B, Nw = len(lens), (c["N"] + 127) // 128 * 128
    M = B * T
    g = _gen(seed)
    x = {}
    if exact:
        x["A"] = _ints((M, K), g)
        x["W"] = _ints((taps, Nw, K), g)
        x["bias"] = _ints((N,), g, -3, 3, torch.float32)
        x["pe"] = _ints((T, 512), g, -16, 16, torch.float32) / 8
        x["alpha"] = 0.5
    else:
        x["A"] = torch.randn(M, K, generator=g, device="cuda").to(torch.bfloat16)
        x["W"] = (torch.randn(taps, Nw, K, generator=g, device="cuda") * 0.05).to(torch.bfloat16)
        x["bias"] = torch.randn(N, generator=g, device="cuda")
        x["pe"] = torch.randn(T, 512, generator=g, device="cuda")
        x["alpha"] = 0.75
    if c.get("resid"):
        dt = torch.bfloat16 if c["resid"] == "bf16" else torch.float32
        x["resid"] = _ints((M, N), g, -4, 4, dt) if exact else torch.randn(M, N, generator=g, device="cuda").to(dt)
    x["lens"] = torch.tensor(lens, dtype=torch.int32, device="cuda")
    return x


def _masks(c, T, B):
    from oracle import philox as px
    M, N = B * T, c["N"]
    m = np.arange(M)
    t, b = m % T, UTT_OFFSET + m // T
    keep_w = px.keep_mask_words(SEED, c["dropw"], t, b, N, P_WORD).cuda() > 0 if c.get("dropw") else None
    keep_b = px.keep_mask_bits(SEED, 0 if "fc1" in c.get("_name", "") else 1, t, b, N).cuda() > 0 if c.get("drop") else None
    return keep_w, keep_b


def _reference(c, x, T, B, exact):
    """(ref, absref): the epilogue in float32 (exact mode) or fp64 (random mode) over the fp64 GEMM, and the same chain on
    absolute values (the scale of the rounding errors in random mode)."""
    N, K, taps = c["N"], c["K"], c.get("taps", 1)
    M, pad = B * T, c.get("taps", 1) // 2

    def conv(a, w):
        ap = F.pad(a.view(B, T, K), (0, 0, pad, pad))
        return sum(ap[:, tap:tap + T].reshape(M, K) @ w[tap, :N].T for tap in range(taps))
    A64, W64 = x["A"].to(F64), x["W"].to(F64)
    keep_w, keep_b = _masks(c, T, B)
    tt = torch.arange(M, device="cuda") % T
    valid = (tt < x["lens"].repeat_interleave(T)).unsqueeze(1)
    out = []
    for absval in (False, True):
        dt = F64 if (absval or not exact) else torch.float32
        acc = conv(A64.abs(), W64.abs()) if absval else conv(A64, W64)
        v = acc.to(dt)
        f = (lambda t: t.to(dt).abs()) if absval else (lambda t: t.to(dt))
        v = v + f(x["bias"])
        if c.get("pe"):
            v = v + abs(x["alpha"]) * f(x["pe"])[tt, :N] if absval else v + x["alpha"] * f(x["pe"])[tt, :N]
        if keep_w is not None:
            v = torch.where(keep_w, v * torch.tensor(DSCALE, dtype=torch.float32).to(dt), torch.zeros_like(v))
        if c.get("resid"):
            v = v + f(x["resid"][:, :N])
        if not absval:
            if c.get("act") == 1:
                v = torch.relu(v)
            elif c.get("act") == 2:
                v = torch.tanh(v)
        if keep_b is not None:
            v = torch.where(keep_b, 2 * v, torch.zeros_like(v))
        if c.get("lens"):
            v = torch.where(valid, v, torch.zeros_like(v))
        out.append(v)
    return out


def _run_site(lib, c, x, T, B, ldo=None, ldr=None, max_ctas=0, offsets=None):
    """Launches the call site's configuration; returns the output buffers (sentinel-filled before the call)."""
    N, K = c["N"], c["K"]
    M = B * T
    offsets = offsets or {}
    kw = dict(A=x["A"], lda=K, W=x["W"], ldw=K, M=M, N=N, K=K, taps=c.get("taps", 1), T=T, act=c.get("act", 0),
              utt_offset=UTT_OFFSET, max_ctas=max_ctas)
    keep = []                                            # tensors that must outlive the call

    def shifted(t, off):                                 # a copy of t starting `off` elements past a 16-byte boundary
        buf = torch.empty(t.numel() + 16, dtype=t.dtype, device="cuda")
        v = buf[off:off + t.numel()]
        v.copy_(t.reshape(-1))
        keep.append(buf)
        return v
    kw["bias"] = shifted(x["bias"], offsets.get("bias", 0))
    if c.get("pe"):
        kw["pe"] = shifted(x["pe"], offsets.get("pe", 0))
        if c["pe"] == "alpha":
            kw["alpha"] = x["alpha"]
        else:
            ap = torch.tensor([x["alpha"]], device="cuda")
            keep.append(ap)
            kw["alpha_ptr"] = ap
    if c.get("lens"):
        kw["lens"] = x["lens"]
    if c.get("drop"):
        kw["drop_site"] = 0 if "fc1" in c["_name"] else 1
        if c["drop"] == "seed":
            kw["seed"] = SEED
        else:
            sp = torch.tensor([SEED], dtype=torch.int64, device="cuda")
            keep.append(sp)
            kw["seed_ptr"] = sp
    if c.get("dropw"):
        sp = torch.tensor([SEED], dtype=torch.int64, device="cuda")
        keep.append(sp)
        kw.update(dropw_site=c["dropw"], dropw_thresh=THRESH, dropw_scale=DSCALE, seed_ptr=sp)
    if c.get("resid"):
        ldr = ldr or c.get("ldr", N)
        r = x["resid"]
        rb = torch.full((M, ldr), 1e4, dtype=r.dtype, device="cuda")        # columns past N: never read
        rb[:, :N] = r
        rb = shifted(rb, offsets.get("resid", 0))
        kw["resid_bf16" if r.dtype == torch.bfloat16 else "resid_f32"] = rb
        kw["ldr"] = ldr
    outs = {}
    if c.get("scatter") == SC_HEAD:
        outs["mel"] = _sentinel((M + 2, 80), torch.float32)
        outs["stop"] = _sentinel((M + 2,), torch.float32)
        kw.update(scatter=SC_HEAD, out_f32=outs["mel"], out2_f32=outs["stop"])
    else:
        ldo = ldo or N
        dt = torch.bfloat16 if c["out"] == "bf16" else torch.float32
        off = offsets.get("out", 0)
        buf = _sentinel(((M + 2) * ldo + 16,), dt)
        keep.append(buf)
        outs["buf"], outs["off"], outs["ldo"] = buf, off, ldo
        outs["out"] = buf[off:off + (M + 2) * ldo].view(M + 2, ldo)
        kw["out_bf16" if dt == torch.bfloat16 else "out_f32"] = outs["out"]
        kw["ldo"] = ldo
    rc = _gemm_epi(lib, **kw)
    assert rc == 0, rc
    torch.cuda.synchronize()
    return outs


def _check_untouched(c, outs, M):
    N = c["N"]
    if "mel" in outs:
        assert _is_sentinel(outs["mel"][M:]) and _is_sentinel(outs["stop"][M:]), "rows past M written"
        return
    o, off = outs["out"], outs["off"]
    assert _is_sentinel(outs["buf"][:off]), "written before the output base"
    assert _is_sentinel(outs["buf"][off + (M + 2) * outs["ldo"]:]), "written past the output buffer"
    assert _is_sentinel(o[M:]), "rows past M written"
    assert _is_sentinel(o[:M, N:]), "columns past N written"


def _result(c, outs, M):
    if "mel" in outs:
        return torch.cat([outs["mel"][:M], outs["stop"][:M, None]], 1)
    return outs["out"][:M, :c["N"]]


def _compare(c, got, ref, absref, exact):
    bf16 = got.dtype == torch.bfloat16
    if exact and c.get("act") != 2:
        want = ref.to(torch.bfloat16) if bf16 else ref
        assert torch.equal(got, want), f"differs at {int((got.float() != want.float()).sum())} of {got.numel()} elements"
        return
    g64, r64 = got.to(F64), ref.to(F64)
    if exact:                                            # tanh: a few fp32 ulp before the rounding
        tol = 8 * 2.0 ** -24 * r64.abs() + 1e-30
    else:
        tol = 1e-4 * absref + 1e-6
    if bf16:
        tol = tol + _bf16_ulp(r64)
    err = (g64 - r64).abs()
    ok = err <= tol
    assert bool(ok.all()), f"{int((~ok).sum())} elements off, max err / tol {float((err / tol).max()):.3g}"


def _site(name):
    return dict(SITES[name], _name=name)


def _gemm_case(lib, name, T, lens, exact, seed, both_forms=True):
    c = _site(name)
    B = len(lens)
    M = B * T
    x = _make_inputs(c, T, lens, exact, seed)
    ref, absref = _reference(c, x, T, B, exact)
    outs = _run_site(lib, c, x, T, B)
    _check_untouched(c, outs, M)
    got = _result(c, outs, M)
    _compare(c, got, ref, absref, exact)
    if both_forms and c.get("scatter", SC_NONE) == SC_NONE:
        # ldo (and ldr) off a multiple of 8: the scalar form only; bit-identical to the vector form
        outs2 = _run_site(lib, c, x, T, B, ldo=c["N"] + 1, ldr=c["N"] + 1 if c.get("resid") else None)
        _check_untouched(c, outs2, M)
        got2 = _result(c, outs2, M)
        diff = _bits(got2) != _bits(got)
        assert not bool(diff.any()), f"scalar and vector forms differ at {int(diff.sum())} elements"
    return c, x, got


@pytest.mark.parametrize("exact", [True, False], ids=["int", "rand"])
@pytest.mark.parametrize("tok", list(TOKENS))
@pytest.mark.parametrize("site", list(SITES))
def test_gemm_site(lib, site, tok, exact):
    T, lens = TOKENS[tok]
    _gemm_case(lib, site, T, lens, exact, seed=list(SITES).index(site) * 10 + list(TOKENS).index(tok) + (0 if exact else 500))


@pytest.mark.parametrize("site", ["enc_conv", "qkv", "wo", "w1", "w2", "train_wo", "prenet_fc1", "post_conv4", "head"])
def test_gemm_site_production_rows(lib, site):
    """B 32 x T 800 = 25 600 rows: the launcher takes 256-column tiles (the small-M cases above take 128) and every CTA
    walks many tiles through the double-buffered accumulator."""
    _gemm_case(lib, site, 800, [800 - 13 * i for i in range(32)], True, seed=800 + list(SITES).index(site))


@pytest.mark.parametrize("site,B,T", [("w1", 8, 512), ("train_wo", 8, 512), ("post_conv4", 8, 512), ("head", 4, 300)])
def test_gemm_max_ctas(lib, site, B, T):
    """The persistent grid capped at 1, 3 and 7 CTAs (the postnet runs capped beside the decode kernel): each CTA walks
    tens to hundreds of tiles, alternating TMEM accumulators, and the result is bit-identical to the uncapped grid."""
    c = _site(site)
    lens = [T - 37 * i for i in range(B)]
    x = _make_inputs(c, T, lens, True, seed=B * T)
    ref, absref = _reference(c, x, T, B, True)
    base = None
    for mc in (0, 1, 3, 7):
        outs = _run_site(lib, c, x, T, B, max_ctas=mc)
        _check_untouched(c, outs, B * T)
        got = _result(c, outs, B * T)
        if base is None:
            _compare(c, got, ref, absref, True)
            base = got.clone()
        else:
            assert torch.equal(_bits(got), _bits(base)), f"max_ctas = {mc} differs from the full grid"


@pytest.mark.parametrize("case", ["out_f32+4", "out_f32+8", "out_bf16+2", "resid_f32+4", "resid_bf16+4", "bias+4", "pe+4",
                                  "mel_after+4"])
def test_gemm_misaligned_operands(lib, case):
    """Operand views that are not 16-byte aligned (a caller's output slice, say) must give the aligned result bit for bit:
    the launcher then keeps the kernel off its 16-byte loads and stores."""
    site, what, nbytes = {
        "out_f32+4": ("wo", "out", 4), "out_f32+8": ("wo", "out", 8), "out_bf16+2": ("qkv", "out", 2),
        "resid_f32+4": ("dgrad_resid", "resid", 4), "resid_bf16+4": ("w2", "resid", 4), "bias+4": ("w1", "bias", 4),
        "pe+4": ("train_enc_proj", "pe", 4), "mel_after+4": ("post_conv4", "out", 4)}[case]
    c = _site(site)
    T, lens = 129, [129, 64, 65]
    B = len(lens)
    for exact in (True, False):
        x = _make_inputs(c, T, lens, exact, seed=len(case) + exact)
        aligned = _result(c, _run_site(lib, c, x, T, B), B * T).clone()
        if exact:
            ref, absref = _reference(c, x, T, B, True)
            _compare(c, aligned, ref, absref, True)
        if what == "out":
            es = 2 if c["out"] == "bf16" else 4
        elif what == "resid":
            es = 2 if c["resid"] == "bf16" else 4
        else:
            es = 4
        outs = _run_site(lib, c, x, T, B, offsets={what: nbytes // es})
        _check_untouched(c, outs, B * T)
        assert torch.equal(_bits(_result(c, outs, B * T)), _bits(aligned)), f"{case}: differs from the aligned run"


# ================================================================================================ cross-K/V scatters
def _kv_inputs(B, S, exact, seed):
    c = dict(N=6144, K=512, _name="cross_kv")
    x = _make_inputs(c, S, [S] * B, exact, seed)
    ref, absref = _reference(c, x, S, B, exact)
    return c, x, ref, absref


@pytest.mark.parametrize("exact", [True, False], ids=["int", "rand"])
@pytest.mark.parametrize("S", [37, 129])
def test_cross_kv_scatter_row_major(lib, S, exact):
    """SC_CROSS_KV (teacher-forced decoder): N = 6 layers x [K | V] x 8 heads x 64 -> cache [6][2][B][8][Lpad][64] bf16.
    Rows S..Lpad-1 of every (layer, kv, b, h) keep what the caller left there (the decode kernel copies 16-row groups)."""
    B, Lpad = 3, (S + 15) // 16 * 16
    c, x, ref, absref = _kv_inputs(B, S, exact, seed=S)
    cache = _sentinel((6, 2, B, 8, Lpad, 64), torch.bfloat16)
    rc = _gemm_epi(lib, A=x["A"], lda=512, W=x["W"], ldw=512, M=B * S, N=6144, K=512, T=S, bias=x["bias"],
                   scatter=SC_CROSS_KV, out_bf16=cache, B=B, Lpad=Lpad)
    assert rc == 0
    torch.cuda.synchronize()
    assert _is_sentinel(cache[:, :, :, :, S:]), "rows past S written"
    got = cache[:, :, :, :, :S].permute(2, 4, 0, 1, 3, 5).reshape(B * S, 6144)        # back to [m][n]
    _compare(dict(c, act=0), got, ref, absref, exact)


@pytest.mark.parametrize("S", [37, 129])
def test_cross_kv_scatter_blocked(lib, S):
    """SC_CROSS_KV_VT (decode kernel): per (layer, b, h) 64-row blocks of four 16-row sub-chunks [K rows | V in MMA
    fragment order], addressed with tts_debug_kv_index.  Every K row and every V fragment element is compared; the rows
    past S of the last block keep the caller's contents."""
    B, nblk = 3, (S + 63) // 64
    Lpad = nblk * 64
    c, x, ref, _ = _kv_inputs(B, S, True, seed=S + 1)
    cache = _sentinel((6, B, 8, nblk, 8192), torch.bfloat16)
    rc = _gemm_epi(lib, A=x["A"], lda=512, W=x["W"], ldw=512, M=B * S, N=6144, K=512, T=S, bias=x["bias"],
                   scatter=SC_CROSS_KV_VT, out_bf16=cache, B=B, Lpad=Lpad)
    assert rc == 0
    torch.cuda.synchronize()
    idx = torch.tensor([[[lib.tts_debug_kv_index(r, d, w) for d in range(64)] for r in range(64)] for w in (0, 1)],
                       dtype=torch.int64, device="cuda")                                 # [kv][row][dim]
    # the expected buffer is built on the bit patterns (a scatter on bf16 values may canonicalise the NaN sentinel)
    want = torch.full((6, B, 8, nblk * 8192), BF16_SENT, dtype=torch.int16, device="cuda")
    r16 = _bits(ref.to(torch.bfloat16)).view(B, S, 6, 2, 8, 64)                            # [b][t][layer][kv][h][d]
    t = torch.arange(S, device="cuda")
    for kv in (0, 1):
        vals = r16[:, :, :, kv].permute(2, 0, 3, 1, 4)                                     # [layer][b][h][t][d]
        flat = (t // 64 * 8192)[:, None] + idx[kv][t % 64]                                 # [t][d] within (layer, b, h)
        want.scatter_(3, flat.reshape(1, 1, 1, S * 64).expand(6, B, 8, S * 64), vals.reshape(6, B, 8, S * 64))
    diff = _bits(cache) != want.view(6, B, 8, nblk, 8192)
    assert not bool(diff.any()), f"blocked cache differs at {int(diff.sum())} elements"


def test_gemm_epi_rejects_what_the_kernel_cannot_do(lib):
    g = _gen(0)
    A = _ints((74, 512), g)
    W = _ints((6144, 512), g)
    cache = torch.zeros(6 * 2 * 2 * 8 * 48 * 64, dtype=torch.bfloat16, device="cuda")
    base = dict(A=A, lda=512, W=W, ldw=512, M=74, N=6144, K=512, T=37, scatter=SC_CROSS_KV, out_bf16=cache, B=2, Lpad=48)
    assert _gemm_epi(lib, **dict(base, Lpad=40)) == -1                 # not a multiple of 16
    assert _gemm_epi(lib, **dict(base, Lpad=32)) == -1                 # < T
    assert _gemm_epi(lib, **dict(base, N=5120 + 512)) == -1            # not a multiple of 1024
    assert _gemm_epi(lib, **dict(base, scatter=SC_CROSS_KV_VT)) == -1  # blocked: Lpad multiple of 64
    assert _gemm_epi(lib, **dict(base, T=36)) == -1                    # M % T
    mel = torch.zeros(74, 80, device="cuda")
    assert _gemm_epi(lib, **dict(base, N=80, scatter=SC_HEAD, out_f32=mel, out2_f32=mel)) == -1
    torch.cuda.synchronize()
    assert not bool(cache.any()) and not bool(mel.any()), "a rejected call wrote"


# ================================================================================================ attention
LOG2E = 1.0 / math.log(2.0)
SCALE_LOG2 = 0.125 * LOG2E


def _attn_call(lib, Q, K, V, O, lse, klens, strides, B, H, Lq, Lk, causal):
    st = (C.c_int64 * 12)(*strides)
    rc = lib.tts_k_attention_strided(C.c_void_p(Q.data_ptr()), C.c_void_p(K.data_ptr()), C.c_void_p(V.data_ptr()),
                                     C.c_void_p(O.data_ptr()), C.c_void_p(lse.data_ptr()) if lse is not None else None,
                                     C.c_void_p(klens.data_ptr()) if klens is not None else None, st, B, H, Lq, Lk, causal, _stream())
    assert rc == 0, rc
    torch.cuda.synchronize()


def _attn_ref(q, k, v, klens, causal):
    """q [B][H][Lq][64], k / v [B][H][Lk][64] (bf16 values) -> O, lse (log2 domain), sum p|v| / sum p, and the largest
    sum_d |q_d k_d| of each row (the scale of the score rounding), all fp64."""
    q, k, v = q.to(F64), k.to(F64), v.to(F64)
    B, H, Lq, Lk = q.shape[0], q.shape[1], q.shape[2], k.shape[2]
    kl = torch.full((B,), Lk, device="cuda") if klens is None else klens.to(torch.int64).clamp(max=Lk)
    j = torch.arange(Lk, device="cuda")
    i = torch.arange(Lq, device="cuda")
    mask = (j[None, :] < kl[:, None])[:, None, None, :]                        # [B][1][1][Lk]
    if causal:
        mask = mask & (j[None, :] <= i[:, None])[None, None]
    s = (q @ k.transpose(-1, -2)) * 0.125
    s = s.masked_fill(~mask, -math.inf)
    mx = s.amax(-1, keepdim=True)
    mx = torch.where(torch.isfinite(mx), mx, torch.zeros_like(mx))
    p = torch.exp(s - mx)
    l = p.sum(-1, keepdim=True)
    safe = torch.where(l > 0, l, torch.ones_like(l))
    O = torch.where(l > 0, (p @ v) / safe, torch.zeros(1, dtype=F64, device="cuda"))
    spv = torch.where(l > 0, (p @ v.abs()) / safe, torch.zeros(1, dtype=F64, device="cuda"))
    lse = torch.where(l[..., 0] > 0, (mx[..., 0] + torch.log(safe[..., 0])) * LOG2E, torch.full_like(l[..., 0], math.inf))
    qk = (q.abs() @ k.abs().transpose(-1, -2)).masked_fill(~mask, 0).amax(-1, keepdim=True)
    return O, lse, spv, qk


def _attn_check(O, lse, ref, Lk):
    """O [B][H][Lq][64] bf16 (any strides), lse [B][H][Lq] against _attn_ref with the bound of the module docstring."""
    Or, lr, spv, qk = ref
    e_s = 64 * 2.0 ** -24 * qk * SCALE_LOG2 * math.log(2.0)          # relative error of p from the score's fp32 rounding
    c = 2.0 ** -8 + 2 * (7.7e-5 + e_s) + Lk * 2.0 ** -23
    tol = c * spv + _bf16_ulp(Or)
    err = (O.to(F64) - Or).abs()
    ok = err <= tol
    assert bool(ok.all()), f"O: {int((~ok).sum())} elements off, max err / tol {float((err / tol).max()):.3g}"
    if lse is not None:
        inf = torch.isinf(lr)
        assert bool((torch.isinf(lse) & (lse > 0))[inf].all()), "lse must be +inf for rows without a visible key"
        tol_l = (7.7e-5 + e_s[..., 0] + Lk * 2.0 ** -24) * LOG2E + 2.0 ** -22 * lr.abs()
        err_l = (lse.to(F64) - lr).abs()
        okl = (err_l <= tol_l) | inf
        assert bool(okl.all()), f"lse: max err / tol {float((err_l / tol_l)[~inf].max()):.3g}"


@pytest.mark.parametrize("causal", [0, 1])
@pytest.mark.parametrize("L,lens", [(37, [37, 20, 1]), (200, [200, 129, 64]), (385, [385, 1, 300])])
def test_attention_packed_qkv(lib, L, lens, causal):
    """Self-attention on the packed QKV GEMM output (ld 1536: Q at +0, K at +512, V at +1024), O at ld 512, as the encoder
    and decoder call it.  Key rows past the lengths hold K of norm 100 and V = 1e4: read once, they would dominate."""
    B, H = len(lens), 8
    g = _gen(L + causal)
    qkv = torch.randn(B, L, 1536, generator=g, device="cuda").to(torch.bfloat16)
    for b, n in enumerate(lens):
        qkv[b, n:, 512:1024] = 12.5
        qkv[b, n:, 1024:] = 1e4
    O = _sentinel((B, L, 512), torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    kl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    s = [L * 1536, 64, 1536] * 3 + [L * 512, 64, 512]
    _attn_call(lib, qkv, qkv[..., 512:], qkv[..., 1024:], O, lse, kl, s, B, H, L, L, causal)
    heads = qkv.view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)                         # [3][B][H][L][64]
    ref = _attn_ref(heads[0], heads[1], heads[2], kl, causal)
    _attn_check(O.view(B, L, H, 64).transpose(1, 2), lse, ref, L)


@pytest.mark.parametrize("T,S,lens", [(37, 37, [37, 20, 1]), (200, 129, [129, 100, 2]), (129, 70, [70, 65, 64])])
def test_attention_cross_from_cache(lib, T, S, lens):
    """Decoder cross-attention (teacher-forced): Q from the [B][T][512] projection, K / V of layer 3 read from the
    row-major cache [6][2][B][8][Spad][64] (k_hs = Spad * 64, Spad > S).  Rows between the lengths and Spad are loud."""
    B, H, Spad = len(lens), 8, (S + 15) // 16 * 16 + 16
    g = _gen(T + S)
    q = torch.randn(B, T, 512, generator=g, device="cuda").to(torch.bfloat16)
    cache = torch.randn(6, 2, B, H, Spad, 64, generator=g, device="cuda").to(torch.bfloat16)
    for b, n in enumerate(lens):
        cache[:, 0, b, :, n:] = 12.5
        cache[:, 1, b, :, n:] = 1e4
    O = _sentinel((B, T, 512), torch.bfloat16)
    lse = torch.empty(B, H, T, device="cuda")
    kl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    kv = [H * Spad * 64, Spad * 64, 64]
    _attn_call(lib, q, cache[3, 0], cache[3, 1], O, lse, kl, [T * 512, 64, 512] + kv + kv + [T * 512, 64, 512], B, H, T, S, 0)
    ref = _attn_ref(q.view(B, T, H, 64).transpose(1, 2), cache[3, 0, :, :, :S], cache[3, 1, :, :, :S], kl, 0)
    _attn_check(O.view(B, T, H, 64).transpose(1, 2), lse, ref, S)


@pytest.mark.parametrize("layer", [0, 5])
def test_attention_cross_training_layout(lib, layer):
    """Training cross-attention: K / V of one layer inside the [B*S][6144] output of the cross-K/V GEMM (ld 6144, K at
    layer * 1024, V at layer * 1024 + 512).  The other layers' columns and the rows past the lengths are loud."""
    B, H, T, S, lens = 3, 8, 150, 90, [90, 45, 1]
    g = _gen(layer)
    q = torch.randn(B, T, 512, generator=g, device="cuda").to(torch.bfloat16)
    kvm = torch.empty(B, S, 6, 2, 512, dtype=torch.bfloat16, device="cuda")
    kvm[:, :, :, 0] = 12.5
    kvm[:, :, :, 1] = 1e4
    kvm[:, :, layer] = torch.randn(B, S, 2, 512, generator=g, device="cuda").to(torch.bfloat16)
    for b, n in enumerate(lens):
        kvm[b, n:, layer, 0] = 12.5
        kvm[b, n:, layer, 1] = 1e4
    kvm = kvm.view(B, S, 6144)
    O = _sentinel((B, T, 512), torch.bfloat16)
    lse = torch.empty(B, H, T, device="cuda")
    kl = torch.tensor(lens, dtype=torch.int32, device="cuda")
    kvs = [S * 6144, 64, 6144]
    _attn_call(lib, q, kvm[..., layer * 1024:], kvm[..., layer * 1024 + 512:], O, lse, kl, [T * 512, 64, 512] + kvs + kvs + [T * 512, 64, 512],
               B, H, T, S, 0)
    kh = kvm.view(B, S, 6, 2, H, 64)[:, :, layer].permute(2, 0, 3, 1, 4)            # [2][B][H][S][64]
    ref = _attn_ref(q.view(B, T, H, 64).transpose(1, 2), kh[0], kh[1], kl, 0)
    _attn_check(O.view(B, T, H, 64).transpose(1, 2), lse, ref, S)


# Rescale: the kernel moves its reference max m (and rescales O and l in TMEM) only when some row of a 32-row warp sees a tile
# maximum more than 8 above m (scaled log2 units; a raw-score jump of 8 / (0.125 log2 e) ~ 44.4).  K carries a per-tile step
# pattern in dimensions 0..3 and small noise elsewhere; each query row picks one pattern with its gain a (scaled jump a * step).
#   pattern 0: steps 0, 1, 2, 3      (a jump at every tile boundary)
#   pattern 1: steps 0, 1, 1, 1      (one jump, at j = 1)
#   pattern 2: steps 0, 0, 0, 1      (one jump, at j = 3)
#   pattern 3: steps 1, 1, 1, 1      (flat)
STEPS = torch.tensor([[0, 1, 2, 3], [0, 1, 1, 1], [0, 0, 0, 1], [1, 1, 1, 1]], dtype=torch.float32)
# per warp: (pattern, scaled jump) of even lanes, of odd lanes, and the tiles at which the warp must rescale
RESCALE_WARPS = [
    ((0, 8.5), (3, 3.0), {1, 2, 3}),      # some rows jump at every boundary, the others never: per-lane mnew
    ((1, 7.5), (1, 7.5), set()),          # just under the threshold: no rescale, P reaches 2^7.5
    ((1, 8.5), (3, 1.0), {1}),            # just over, at j = 1
    ((2, 9.0), (1, 7.5), {3}),            # late jump beside rows that stay 7.5 above their reference
]


def _rescale_inputs(seed):
    B, H, Lq, Lk = 1, 2, 128, 512
    g = _gen(seed)
    q = torch.randn(B, H, Lq, 64, generator=g, device="cuda") * 0.1
    k = torch.randn(B, H, Lk, 64, generator=g, device="cuda") * 0.1
    k[..., :4] = STEPS.cuda().T.repeat_interleave(128, 0)                             # [Lk][4]: step of each key's tile
    q[..., :4] = 0
    for w, (even, odd, _) in enumerate(RESCALE_WARPS):
        for lane in range(32):
            pat, jump = even if lane % 2 == 0 else odd
            q[..., w * 32 + lane, pat] = jump / SCALE_LOG2
    v = torch.randn(B, H, Lk, 64, generator=g, device="cuda")
    return q.to(torch.bfloat16), k.to(torch.bfloat16), v.to(torch.bfloat16)


def _rescale_premise(q, k):
    """The kernel's decision, replayed in fp64 on the bf16 inputs: per warp and tile, does some row's tile max exceed the
    warp's reference by more than 8?  Returns {warp: set of tiles that rescale} and whether every rescaling warp also has
    rows that do not jump there."""
    s = (q.to(F64) @ k.to(F64).transpose(-1, -2)) * SCALE_LOG2                        # [B][H][Lq][Lk], scaled log2 units
    tmax = s.view(*s.shape[:3], 4, 128).amax(-1)                                       # [B][H][Lq][tile]
    fired, mixed = {}, True
    for w in range(4):
        rows = tmax[:, :, w * 32:(w + 1) * 32]                                         # [B][H][32][tile]
        m = torch.full(rows.shape[:3], -math.inf, dtype=F64, device=rows.device)
        tiles = set()
        for j in range(4):
            over = rows[..., j] > m + 8
            if bool(over.any()):
                if j > 0:
                    tiles.add(j)
                    mixed &= bool((~over).any())
                m = torch.maximum(m, rows[..., j])
        fired[w] = tiles
    return fired, mixed


def test_attention_rescale(lib):
    """O and l rescaled in TMEM when a row's tile max jumps by more than 2^8 (at j = 1, 2, 3, with other rows of the warp not
    jumping), and left alone for a jump of 7.5 (P = 2^7.5 in bf16).  The test first checks its own premise on the host."""
    q, k, v = _rescale_inputs(3)
    fired, mixed = _rescale_premise(q, k)
    for w, (_, _, want) in enumerate(RESCALE_WARPS):
        assert fired[w] == want, f"premise: warp {w} rescales at tiles {fired[w]}, expected {want}"
    assert mixed, "premise: every rescaling warp must also hold rows that do not jump"
    B, H, Lq, Lk = 1, 2, 128, 512
    O = _sentinel((B, H, Lq, 64), torch.bfloat16)
    lse = torch.empty(B, H, Lq, device="cuda")
    s = [H * Lq * 64, Lq * 64, 64, H * Lk * 64, Lk * 64, 64, H * Lk * 64, Lk * 64, 64, H * Lq * 64, Lq * 64, 64]
    _attn_call(lib, q, k, v, O, lse, None, s, B, H, Lq, Lk, 0)
    _attn_check(O, lse, _attn_ref(q, k, v, None, 0), Lk)


@pytest.mark.parametrize("causal", [0, 1])
def test_attention_empty_and_clamped_keys(lib, causal):
    """klens = 0: no visible key, O = 0 and lse = +inf.  klens > Lk: clamped to Lk (the rows past Lk in memory are loud and
    lie outside the tensor maps; a key count past Lk would add zero-filled keys to l)."""
    B, H, L = 3, 8, 200
    g = _gen(7 + causal)
    buf = torch.randn(B, L + 64, 1536, generator=g, device="cuda").to(torch.bfloat16)
    buf[:, L:, 512:1024] = 12.5
    buf[:, L:, 1024:] = 1e4
    qkv = buf[:, :L]
    kl = torch.tensor([0, L + 100, 77], dtype=torch.int32, device="cuda")
    O = _sentinel((B, L, 512), torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    s = [(L + 64) * 1536, 64, 1536] * 3 + [L * 512, 64, 512]
    _attn_call(lib, qkv, qkv[..., 512:], qkv[..., 1024:], O, lse, kl, s, B, H, L, L, causal)
    assert not bool(O[0].float().any()), "klens = 0: O must be zero"
    assert bool((torch.isinf(lse[0]) & (lse[0] > 0)).all()), "klens = 0: lse must be +inf"
    heads = qkv.reshape(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    ref = _attn_ref(heads[0], heads[1], heads[2], kl, causal)
    _attn_check(O.view(B, L, H, 64).transpose(1, 2), lse, ref, L)


@pytest.mark.parametrize("L", [129, 255, 385])
def test_attention_causal_tile_edges(lib, L):
    """Causal with Lq % 128 in {1, 127}: the last query tile is one row / one row short; the diagonal key of every row is
    visible (row 0 sees exactly one key)."""
    B, H = 2, 8
    g = _gen(L)
    qkv = torch.randn(B, L, 1536, generator=g, device="cuda").to(torch.bfloat16)
    O = _sentinel((B, L, 512), torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    kl = torch.tensor([L, L - 1], dtype=torch.int32, device="cuda")
    s = [L * 1536, 64, 1536] * 3 + [L * 512, 64, 512]
    _attn_call(lib, qkv, qkv[..., 512:], qkv[..., 1024:], O, lse, kl, s, B, H, L, L, 1)
    heads = qkv.view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4)
    ref = _attn_ref(heads[0], heads[1], heads[2], kl, 1)
    _attn_check(O.view(B, L, H, 64).transpose(1, 2), lse, ref, L)
    # row 0 attends to key 0 only: O = bf16(V[0]) exactly
    assert torch.equal(O.view(B, L, H, 64)[:, 0], qkv.view(B, L, 3, H, 64)[:, 0, 2])


def test_attention_strided_rejects_unaligned_strides(lib):
    x = torch.zeros(2, 64, 1536, dtype=torch.bfloat16, device="cuda")
    O = _sentinel((2, 64, 512), torch.bfloat16)
    for i in range(12):
        s = [64 * 1536, 64, 1536] * 3 + [64 * 512, 64, 512]
        s[i] += 4
        st = (C.c_int64 * 12)(*s)
        assert lib.tts_k_attention_strided(C.c_void_p(x.data_ptr()), C.c_void_p(x.data_ptr()), C.c_void_p(x.data_ptr()),
                                           C.c_void_p(O.data_ptr()), None, None, st, 2, 8, 64, 64, 0, _stream()) == -1
    torch.cuda.synchronize()
    assert _is_sentinel(O)
