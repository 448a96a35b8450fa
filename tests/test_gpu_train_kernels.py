"""Per-kernel parity of the training step's own kernels on a real B200 (pytest -m gpu): weight gradient (tcgen05, split-K),
input gradient (packed transposed weights + GEMM), masked batch-statistics BatchNorm forward / backward, LayerNorm backward,
loss and head gradient, word-dropout and embedding backward.  Each is called through its tts_k_* entry point, which launches
exactly what tts_train_step launches, and compared with an fp64 computation on the same (bf16-rounded) inputs.  Dropout masks
come from oracle/philox.py.

The tensor-core cases with small-integer inputs (|v| <= 2) must match EXACTLY: every product and every partial sum is an
integer below 2^17, so fp32 accumulation is exact whatever the split-K or atomic order.  A dropped token block, a misplaced
conv tap or a lost bias split then fails on any shape instead of hiding inside a tolerance."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

F64 = torch.float64
EPS32 = 2.0 ** -24


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from transformer_tacotron2_b200 import _lib
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    return _lib.load()


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _seed_dev(seed):
    return torch.tensor([seed], dtype=torch.int64, device="cuda")        # read by the kernels as a uint64


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _ints(shape, g):
    """Integers in [-2, 2]: exact in bf16; products and sums below 2^24 are exact in fp32."""
    return torch.randint(-2, 3, shape, generator=g, device="cuda").to(torch.bfloat16)


def _valid(lens, T):
    return torch.arange(T, device=lens.device)[None, :] < lens[:, None]             # [B][T] bool


def _bf16_ulp(x):
    """One bf16 ulp at |x| (8 significant bits); the smallest normal's ulp for zero."""
    a = x.abs().clamp(min=2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


# ================================================================================================ weight gradient
# (Cout, Cin, taps, ldy, ldx) of the training step (train.cuh, train_backward)
WG_LAYERS = {
    "qkv": (1536, 512, 1, 1536, 512),
    "ffn1": (2048, 512, 1, 2048, 512),
    "ffn2": (512, 2048, 1, 512, 2048),
    "cross_kv": (6144, 512, 1, 6144, 512),
    "fc1": (256, 80, 1, 256, 96),
    "head": (81, 512, 1, 128, 512),
    "enc_conv": (512, 512, 5, 512, 512),
    "post_conv0": (512, 80, 5, 512, 96),
    "post_conv4": (80, 512, 5, 80, 512),
}
# token layouts: (T, lens) with nb = len(lens); lens None = every row valid.  A linear layer sees all rows as one "utterance"
# (T = M, nb = 1), as in the training step.
WG_TOKENS = {
    "T1": (1, None),
    "T37": (37, None),                       # M < 64
    "T129x3": (129, [129, 100, 1]),
    "T150x5": (150, [150, 77, 1, 149, 64]),  # ragged, zero rows past each length
}


def _wgrad_ref(dY, X, Cout, Cin, taps, T, nb):
    """fp64 dW [Cout][Cin * taps] (element k * taps + tap) and db [Cout]; X rows shifted by tap - taps // 2 inside each
    utterance, zero outside."""
    pad = taps // 2
    dy = dY[:, :Cout].to(F64)
    x = X[:, :Cin].to(F64).view(nb, T, Cin)
    xp = F.pad(x, (0, 0, pad, pad))
    dW = torch.stack([dy.T @ xp[:, tap:tap + T].reshape(nb * T, Cin) for tap in range(taps)], dim=-1)
    return dW.reshape(Cout, Cin * taps), dy.sum(0)


def _wgrad_abs_ref(dY, X, Cout, Cin, taps, T, nb):
    return _wgrad_ref(dY.abs(), X.abs(), Cout, Cin, taps, T, nb)


def _run_wgrad(lib, dY, ldy, Cout, X, ldx, Cin, taps, T, nb, dW, db):
    rc = lib.tts_k_wgrad(_p(dY), ldy, Cout, _p(X), ldx, Cin, taps, T, nb, _p(dW), _p(db), _stream())
    assert rc == 0
    torch.cuda.synchronize()


def _wgrad_inputs(g, Cout, Cin, ldy, ldx, M, row_valid, exact):
    if exact:
        dY, X = _ints((M, ldy), g), _ints((M, ldx), g)
    else:
        dY = torch.randn(M, ldy, generator=g, device="cuda").to(torch.bfloat16)
        X = torch.randn(M, ldx, generator=g, device="cuda").to(torch.bfloat16)
    if row_valid is not None:                # training: rows past each length are zero in both operands
        dY, X = dY * row_valid[:, None], X * row_valid[:, None]
    # columns past Cout / Cin (the head's 81..127, fc1's 80..95) are read by nobody: make them loud
    dY[:, Cout:] = 100
    X[:, Cin:] = 100
    return dY.contiguous(), X.contiguous()


def _wgrad_case(lib, Cout, Cin, taps, ldy, ldx, T, nb, row_valid, exact, seed, with_bias=True, dw_offset=0):
    g = _gen(seed)
    dY, X = _wgrad_inputs(g, Cout, Cin, ldy, ldx, T * nb, row_valid, exact)
    # accumulate semantics: dW and db start non-zero (integers, so the exact cases stay exact)
    buf = torch.empty(Cout * Cin * taps + dw_offset, device="cuda")
    dW = buf[dw_offset:].view(Cout, Cin * taps)
    dW.copy_(torch.randint(-3, 4, dW.shape, generator=g, device="cuda").float())
    db = torch.randint(-3, 4, (Cout,), generator=g, device="cuda").float() if with_bias else None
    dW0, db0 = dW.clone().to(F64), (db.clone().to(F64) if with_bias else None)
    _run_wgrad(lib, dY, ldy, Cout, X, ldx, Cin, taps, T, nb, dW, db)
    ref_w, ref_b = _wgrad_ref(dY, X, Cout, Cin, taps, T, nb)
    ref_w = ref_w + dW0
    if exact:
        assert torch.equal(dW.to(F64), ref_w), f"dW differs at {int((dW.to(F64) != ref_w).sum())} elements"
        if with_bias:
            assert torch.equal(db.to(F64), ref_b + db0)
        return
    abs_w, abs_b = _wgrad_abs_ref(dY, X, Cout, Cin, taps, T, nb)
    err = (dW.to(F64) - ref_w).abs()
    tol = 1e-4 * abs_w + 1e-6
    assert bool((err <= tol).all()), f"dW: max err / tol {float((err / tol).max()):.3g}"
    if with_bias:
        err_b = (db.to(F64) - ref_b - db0).abs()
        assert bool((err_b <= 1e-4 * abs_b + 1e-6).all()), float(err_b.max())


def _rows_valid(lens, T):
    return None if lens is None else _valid(torch.tensor(lens, device="cuda"), T).reshape(-1)


def _layout(layer, tok):
    Cout, Cin, taps, ldy, ldx = WG_LAYERS[layer]
    T, lens = WG_TOKENS[tok]
    nb = len(lens) if lens is not None else 1
    row_valid = _rows_valid(lens, T)
    if taps == 1:                            # a linear layer's weight gradient runs over all M rows as one slab
        T, nb = T * nb, 1
    return Cout, Cin, taps, ldy, ldx, T, nb, row_valid


@pytest.mark.parametrize("exact", [True, False], ids=["int", "rand"])
@pytest.mark.parametrize("tok", list(WG_TOKENS))
@pytest.mark.parametrize("layer", list(WG_LAYERS))
def test_wgrad(lib, layer, tok, exact):
    Cout, Cin, taps, ldy, ldx, T, nb, row_valid = _layout(layer, tok)
    _wgrad_case(lib, Cout, Cin, taps, ldy, ldx, T, nb, row_valid, exact, seed=list(WG_LAYERS).index(layer) * 100 + list(WG_TOKENS).index(tok))


@pytest.mark.parametrize("exact", [True, False], ids=["int", "rand"])
@pytest.mark.parametrize("layer,T,nb", [("qkv", 25600, 1), ("ffn1", 25600, 1), ("ffn2", 25600, 1), ("cross_kv", 25600, 1),
                                        ("head", 25600, 1), ("fc1", 25600, 1),
                                        ("enc_conv", 800, 32), ("post_conv0", 800, 32), ("post_conv4", 800, 32)])
def test_wgrad_production_tokens(lib, layer, T, nb, exact):
    """B 32 x T 800 = 25 600 decoder tokens, the measured training shape: the split-K heuristic picks its production split
    counts, so every split's token range and its share of the bias gradient are checked."""
    Cout, Cin, taps, ldy, ldx = WG_LAYERS[layer]
    row_valid = _rows_valid([800 - 13 * i for i in range(nb)], T) if taps > 1 else None
    _wgrad_case(lib, Cout, Cin, taps, ldy, ldx, T, nb, row_valid, exact, seed=T + nb + Cout)


@pytest.mark.parametrize("taps,T,nb", [(1, 129, 1), (5, 37, 3), (5, 150, 2)])
def test_wgrad_cin_not_multiple_of_4(lib, taps, T, nb):
    """Cin = 90 (ldx 96): no TMA reduce-add, the scalar-atomic epilogue."""
    for exact in (True, False):
        _wgrad_case(lib, 256, 90, taps, 256, 96, T, nb, None, exact, seed=90 + T)


@pytest.mark.parametrize("layer", ["qkv", "head", "fc1", "enc_conv"])
def test_wgrad_without_bias(lib, layer):
    Cout, Cin, taps, ldy, ldx, T, nb, row_valid = _layout(layer, "T150x5")
    _wgrad_case(lib, Cout, Cin, taps, ldy, ldx, T, nb, row_valid, True, seed=11, with_bias=False)


@pytest.mark.parametrize("layer,T", [("qkv", 150), ("head", 1), ("ffn2", 2000), ("fc1", 37)])
def test_wgrad_dw_not_16_byte_aligned(lib, layer, T):
    """dW one float past a 16-byte boundary: the TMA reduce-add cannot describe it, so the partial tiles go through the
    scalar atomics (no vector reduction to a misaligned address)."""
    Cout, Cin, taps, ldy, ldx = WG_LAYERS[layer]
    for exact in (True, False):
        _wgrad_case(lib, Cout, Cin, taps, ldy, ldx, T, 1, None, exact, seed=T, dw_offset=1)


@pytest.mark.parametrize("layer,T,lens", [("enc_conv", 150, [150, 64, 2, 129, 65]), ("post_conv0", 130, [130, 1, 66]),
                                          ("post_conv4", 800, [800, 799, 64, 63])])
def test_wgrad_conv_utterance_boundaries(lib, layer, T, lens):
    """dY non-zero only at t in {0, 1, 63, 64, T-2, T-1} inside each length, X non-zero everywhere (also past the lengths):
    the taps at t < 2 and t > T - 3 must see zero padding, never the neighbouring utterance's rows."""
    Cout, Cin, taps, ldy, ldx = WG_LAYERS[layer]
    nb = len(lens)
    g = _gen(T + nb)
    dY = _ints((nb * T, ldy), g).view(nb, T, ldy)
    X = _ints((nb * T, ldx), g)
    X[X == 0] = 1
    probe = torch.zeros(nb, T, dtype=torch.bool, device="cuda")
    for b, L in enumerate(lens):
        for t in (0, 1, 63, 64, T - 2, T - 1):
            if 0 <= t < L:
                probe[b, t] = True
    dY = (dY * probe[..., None]).reshape(nb * T, ldy).contiguous()
    dW = torch.zeros(Cout, Cin * taps, device="cuda")
    db = torch.zeros(Cout, device="cuda")
    _run_wgrad(lib, dY, ldy, Cout, X, ldx, Cin, taps, T, nb, dW, db)
    ref_w, ref_b = _wgrad_ref(dY, X, Cout, Cin, taps, T, nb)
    assert torch.equal(dW.to(F64), ref_w), f"dW differs at {int((dW.to(F64) != ref_w).sum())} elements"
    assert torch.equal(db.to(F64), ref_b)


# ================================================================================================ input gradient
def _dgrad_case(lib, N, K, taps, ldy, Kdy, T, lens, exact, out_bf16, ldo, seed):
    nb = len(lens)
    M = nb * T
    g = _gen(seed)
    if exact:
        W = torch.randint(-2, 3, (N, K, taps), generator=g, device="cuda").float()
        dY = _ints((M, ldy), g)
    else:
        W = torch.randn(N, K, taps, generator=g, device="cuda") * 0.05
        dY = torch.randn(M, ldy, generator=g, device="cuda").to(torch.bfloat16)
    valid = _valid(torch.tensor(lens, device="cuda"), T).reshape(M, 1)
    dY = dY * valid                                      # the gradient wrt a conv output is zero past each length
    dY[:, N:] = 7                                        # head: columns 81..127 of dhead meet the zero rows of the packed weight
    dY = dY.contiguous()
    Wq = W.to(torch.bfloat16).to(F64)                    # the kernel packs bf16(W)
    scratch = torch.empty(taps * ((K + 127) // 128 * 128) * ((N + 63) // 64 * 64), dtype=torch.bfloat16, device="cuda")
    out = torch.full((M, ldo), -3.0, dtype=torch.bfloat16 if out_bf16 else torch.float32, device="cuda")
    rc = lib.tts_k_dgrad(_p(W), N, K, taps, _p(dY), ldy, Kdy, M, T, None if out_bf16 else _p(out), _p(out) if out_bf16 else None,
                         ldo, _p(scratch), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    dy = dY[:, :N].to(F64)
    if taps == 1:
        ref, ref_abs = dy @ Wq[:, :, 0], dy.abs() @ Wq[:, :, 0].abs()
    else:
        # dX[t] = sum_tap dY[t + pad - tap] . W[:, :, tap] as tap-shifted matrix products: exact in fp64 on integers, which
        # torch's fp64 conv1d_input on CUDA is not (its convolution algorithms leave ~1e-14 residues)
        pad = taps // 2

        def conv_in(d, w):
            dp = F.pad(d.view(nb, T, N), (0, 0, pad, pad))
            return sum(dp[:, 2 * pad - tap:2 * pad - tap + T].reshape(M, N) @ w[:, :, tap] for tap in range(taps))
        ref, ref_abs = conv_in(dy, Wq), conv_in(dy.abs(), Wq.abs())
        via_torch = torch.nn.grad.conv1d_input((nb, K, T), Wq, dy.view(nb, T, N).transpose(1, 2), padding=pad).transpose(1, 2).reshape(M, K)
        assert torch.allclose(via_torch, ref, rtol=1e-12, atol=1e-12 * float(ref_abs.max()))
    got = out[:, :K].to(F64)
    assert bool((out[:, K:].float() == -3.0).all()), "columns past K written"
    if exact:
        want = ref.to(torch.bfloat16).to(F64) if out_bf16 else ref
        assert torch.equal(got, want), f"dX differs at {int((got != want).sum())} elements"
        return
    tol = 1e-4 * ref_abs + 1e-6 + (_bf16_ulp(ref) if out_bf16 else 0.0)
    err = (got - ref).abs()
    assert bool((err <= tol).all()), f"dX: max err / tol {float((err / tol).max()):.3g}"


DG_LENS = {1: [1, 1, 1], 5: [5, 1, 3, 5], 37: [37, 20, 1, 36, 2], 129: [129, 64, 65], 300: [300, 299, 1, 150, 257]}


@pytest.mark.parametrize("exact", [True, False], ids=["int", "rand"])
@pytest.mark.parametrize("T", list(DG_LENS))
@pytest.mark.parametrize("N,K,ldo", [(80, 512, 512), (512, 80, 96), (512, 512, 512)], ids=["post_conv4", "post_conv0", "conv512"])
def test_dgrad_conv(lib, N, K, ldo, T, exact):
    """conv5 input gradient through the transposed, tap-reversed packed weights (bf16 output, as the training step writes it).
    N = 80 makes the reduction 80 (not a multiple of 64); K = 80 makes the output 80 columns wide inside a 96-wide buffer."""
    _dgrad_case(lib, N, K, 5, N, N, T, DG_LENS[T], exact, True, ldo, seed=N + K + T)
    if exact:
        _dgrad_case(lib, N, K, 5, N, N, T, DG_LENS[T], exact, False, ldo, seed=N + K + T + 1)


@pytest.mark.parametrize("exact", [True, False], ids=["int", "rand"])
@pytest.mark.parametrize("T,lens", [(37, [37, 5]), (800, [800, 1, 640])])
def test_dgrad_head(lib, T, lens, exact):
    """Heads (taps = 1): N = 81, reduction over the 128 columns of dhead; packed weight rows 81..127 must be zero."""
    _dgrad_case(lib, 81, 512, 1, 128, 128, T, lens, exact, False, 512, seed=T)


# ================================================================================================ masked BatchNorm
def _bn_case(lib, C, act, site, lens, T, seed, utt_offset=0, mean=0.0, std=1.0, dout_bf16=True):
    from oracle import philox as px
    from oracle.transformer_tts import masked_batchnorm
    B = len(lens)
    M = B * T
    g = _gen(seed)
    lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
    valid = _valid(lens_t, T)                                              # [B][T]
    x = torch.randn(M, C, generator=g, device="cuda") * std + mean
    x[~valid.reshape(M)] = 1e4                                             # padded rows: garbage the statistics must skip
    gamma = torch.rand(C, generator=g, device="cuda") + 0.5
    beta = torch.randn(C, generator=g, device="cuda") * 0.5
    rm0 = torch.randn(C, generator=g, device="cuda")
    rv0 = torch.rand(C, generator=g, device="cuda") + 0.5
    eps, seed_v = 1e-5, 0x1234_5678_9ABC + seed
    seed_d = _seed_dev(seed_v)
    ldo = C + 16
    stat = torch.full((1024,), 777.0, device="cuda")
    out16 = torch.full((M, ldo), -3.0, dtype=torch.bfloat16, device="cuda")   # sentinel in the columns C..ldo-1
    out32 = torch.empty(M, C, device="cuda")
    rm, rv = rm0.clone(), rv0.clone()
    rc = lib.tts_k_bn_train_fwd(_p(x), B, T, C, _p(lens_t), _p(stat), _p(gamma), _p(beta), eps, act, site, _p(seed_d), utt_offset,
                                _p(out16), ldo, _p(out32), _p(rm), _p(rv), _stream())
    assert rc == 0
    torch.cuda.synchronize()

    # ---- fp64 reference: the oracle's masked BatchNorm on [B][C][T], then activation, p = 0.5 dropout, length mask
    bn = torch.nn.BatchNorm1d(C, eps=eps, momentum=0.1).to(F64).cpu()
    with torch.no_grad():
        bn.weight.copy_(gamma.cpu()); bn.bias.copy_(beta.cpu()); bn.running_mean.copy_(rm0.cpu()); bn.running_var.copy_(rv0.cpu())
    x64 = x.cpu().to(F64).view(B, T, C).transpose(1, 2).requires_grad_(True)
    mask = valid.cpu().to(F64)[:, None, :]
    yb = masked_batchnorm(bn, x64, mask, training=True)                   # [B][C][T]
    y = torch.relu(yb) if act == 1 else torch.tanh(yb) if act == 2 else yb
    keep = torch.ones(B, T, C, dtype=F64)
    if site >= 0:
        keep = px.keep_mask_bits(seed_v, site, torch.arange(T)[None, :].numpy(), (utt_offset + torch.arange(B))[:, None].numpy(), C).to(F64)
        y = y * keep.transpose(1, 2) * 2.0
    y = y * mask
    ref = y.transpose(1, 2).reshape(M, C).detach()

    n = float(sum(lens))
    xv = x.cpu().to(F64)[valid.reshape(M).cpu()]
    m64 = xv.mean(0)
    st = stat.cpu().to(F64)
    # stat: sums to 1e-5; the centred sum of squares is checked around the kernel's own mean (the second pass's input), so
    # an imprecise variance cannot hide behind a first-pass rounding
    assert torch.allclose(st[:C], xv.sum(0), rtol=1e-5, atol=1e-5 * float(xv.abs().sum(0).max())), "stat: sums"
    mk = (stat[:C].cpu() / torch.tensor(n, dtype=torch.float32)).to(F64)     # the mean as the kernel forms it (fp32)
    assert torch.allclose(st[C:2 * C], ((xv - mk) ** 2).sum(0), rtol=1e-5, atol=0.0), "stat: centred sum of squares"
    assert torch.allclose(st[C:2 * C], ((xv - m64) ** 2).sum(0), rtol=1e-3, atol=0.0), "stat: variance vs the fp64 mean"
    # running statistics (unbiased variance)
    assert torch.allclose(rm.cpu().to(F64), bn.running_mean, rtol=1e-5, atol=1e-6)
    assert torch.allclose(rv.cpu().to(F64), bn.running_var, rtol=1e-5, atol=1e-6)

    # out32 to 1e-4, plus the fp32 conditioning of the fused scale / shift x * sc + sh and of the kernel's mean / rstd
    # (large-mean data: |x * sc| >> |y| loses digits in ANY fp32 evaluation of that form)
    var64 = ((xv - m64) ** 2).mean(0)
    rstd64 = (var64 + eps) ** -0.5
    rstdk = (st[C:2 * C] / n + eps) ** -0.5
    sc = rstd64 * gamma.cpu().to(F64)
    sh = beta.cpu().to(F64) - m64 * sc
    xa = x.cpu().to(F64)
    cond = (xa * sc).abs() + sh.abs() + sc.abs() * (mk - m64).abs() + (ref.abs() + beta.cpu().to(F64).abs()) * ((rstdk - rstd64).abs() / rstd64)
    tol_y = 2.0 * (8 * EPS32 * cond + 1e-4 * ref.abs()) + 1e-6
    vm = valid.reshape(M).cpu()
    got32 = out32.cpu().to(F64)
    err = (got32 - ref).abs()
    assert bool((err[vm] <= tol_y[vm]).all()), f"out32: max err / tol {float((err[vm] / tol_y[vm]).max()):.3g}"
    assert bool((out32.cpu()[~vm] == 0).all()), "out32: padded rows must be exactly zero"
    assert torch.equal(out16[:, :C], out32.to(torch.bfloat16)), "out16 must be bf16(out32)"
    assert bool((out16[:, C:].float() == -3.0).all()), "out16: columns past C written"

    # ---- backward: dout (fp32 [M][C], or bf16 with row stride ldd), reference by autograd through the same oracle graph
    ldd = C + 8
    dout_full = torch.randn(M, ldd, generator=g, device="cuda")
    dout_full[~valid.reshape(M)] = 0.0                     # the training step's upstream gradient is zero past the lengths
    if dout_bf16:
        dout_dev = dout_full.to(torch.bfloat16)
    else:
        dout_dev = dout_full[:, :C].contiguous()
        ldd = C
    d64 = dout_dev[:, :C].cpu().to(F64)
    y.backward(d64.view(B, T, C).transpose(1, 2))
    ref_dx = x64.grad.transpose(1, 2).reshape(M, C)
    ref_dg, ref_db = bn.weight.grad, bn.bias.grad
    dgam = torch.zeros(C, device="cuda")
    dbet = torch.zeros(C, device="cuda")
    ldx = C + 4
    dx = torch.full((M, ldx), -5.0, dtype=torch.bfloat16, device="cuda")
    rc = lib.tts_k_bn_train_bwd(_p(dout_dev), int(dout_bf16), ldd, _p(x), B, T, C, _p(lens_t), _p(stat), _p(gamma), _p(beta), eps, act, site,
                                _p(seed_d), utt_offset, _p(dgam), _p(dbet), _p(dx), ldx, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    # gradient wrt the BN output and xhat, fp64: the scale of every sum below
    xh = ((xa - m64) * rstd64).view(B, T, C)
    ybt = yb.detach().transpose(1, 2)
    gb = d64.view(B, T, C) * (keep * 2.0 if site >= 0 else 1.0)
    if act == 1:
        gb = gb * (ybt > 0)
    elif act == 2:
        gb = gb * (1 - torch.tanh(ybt) ** 2)
    gb = gb * valid.cpu()[..., None]
    # a ReLU whose input is within rounding of 0 may go either way in fp32: those elements are excused below
    flip = (ybt.abs() < 1e-5 * (1 + cond.view(B, T, C))) & valid.cpu()[..., None] if act == 1 else torch.zeros(B, T, C, dtype=torch.bool)
    dxh = (xa - mk).view(B, T, C) * rstdk - xh                              # the kernel's xhat minus the fp64 one
    slack = (d64.view(B, T, C).abs() * 2 * flip).sum((0, 1))
    # tanh' moves by at most 0.77 x the shift of its input, gamma * (xhat_kernel - xhat)
    dact = (d64.view(B, T, C).abs() * 2 * gamma.cpu().to(F64).abs() * dxh.abs() * valid.cpu()[..., None]) if act == 2 else torch.zeros_like(gb)
    tol_db = 1e-4 * gb.abs().sum((0, 1)) + slack + dact.sum((0, 1)) + 1e-6
    tol_dg = (1e-4 * (gb * xh).abs().sum((0, 1)) + (gb.abs() * dxh.abs()).sum((0, 1)) + slack * xh.abs().amax((0, 1))
              + (dact * xh.abs()).sum((0, 1)) + 1e-6)
    assert bool(((dbet.cpu().to(F64) - ref_db).abs() <= tol_db).all()), "dbeta"
    assert bool(((dgam.cpu().to(F64) - ref_dg).abs() <= tol_dg).all()), "dgamma"
    # dx within one bf16 ulp of the fp64 value, plus the fp32 cancellation in g - mean(g) - xhat mean(g xhat)
    ga = gamma.cpu().to(F64)
    mg, mgx = gb.sum((0, 1)) / n, (gb * xh).sum((0, 1)) / n
    scale = (ga * rstd64).abs()
    cond_dx = scale * (gb.abs() + mg.abs() + (xh * mgx).abs())
    # the errors allowed in dbeta / dgamma reach dx through mean(g) and mean(g * xhat) unscaled (first-order terms x 2)
    tol_dx = (_bf16_ulp(ref_dx.view(B, T, C)) + 1e-5 * cond_dx + 2 * scale * (dact + mgx.abs() * dxh.abs() + tol_db / n + xh.abs() * tol_dg / n) + 2 * ref_dx.view(B, T, C).abs() * ((rstdk - rstd64).abs() / rstd64))
    got_dx = dx[:, :C].cpu().to(F64).view(B, T, C)
    err_dx = (got_dx - ref_dx.view(B, T, C)).abs()
    ok = (err_dx <= tol_dx) | flip
    assert bool(ok.all()), f"dx: {int((~ok).sum())} elements off, max err / tol {float((err_dx / tol_dx)[~flip].max()):.3g}"
    assert bool((got_dx[~valid.cpu()] == 0).all()), "dx: padded rows must be exactly zero"
    assert bool((dx[:, C:].float() == -5.0).all()), "dx: columns past C written"


BN_LENS = {
    "ragged": (150, [150, 1, 77, 149, 64]),          # M = 750 < 592 x rows: some statistics row chunks are empty
    "single": (40, [1]),                             # one valid position in the whole batch (n = 1)
    # 16 000 rows > 1184 blocks x row lanes (2 at C = 512, 12 at C = 80): the element-wise grid-stride loops wrap
    "long": (800, [800, 700, 1, 650, 799, 512, 433, 800, 9, 640, 777, 800, 64, 63, 800, 2, 555, 800, 321, 799]),
}


@pytest.mark.parametrize("layout", list(BN_LENS))
@pytest.mark.parametrize("C,act,site", [(512, 1, 2), (512, 2, 5), (80, 0, 9), (80, 0, -1), (512, 0, -1), (80, 2, 7)])
def test_bn_train(lib, C, act, site, layout):
    T, lens = BN_LENS[layout]
    _bn_case(lib, C, act, site, lens, T, seed=C + act + T, utt_offset=0 if site < 0 else 13, dout_bf16=(C == 512))


@pytest.mark.parametrize("dout_bf16", [True, False])
def test_bn_train_dout_dtypes(lib, dout_bf16):
    _bn_case(lib, 512, 1, 3, [37, 20, 5], 37, seed=5, utt_offset=7, dout_bf16=dout_bf16)
    _bn_case(lib, 80, 2, 5, [37, 20, 5], 37, seed=6, utt_offset=0, dout_bf16=dout_bf16)


@pytest.mark.parametrize("C,act", [(512, 2), (80, 0)])
def test_bn_train_large_mean_small_spread(lib, C, act):
    """mean 100, std 1e-2: the centred second pass keeps the variance; a one-pass E[x^2] - E[x]^2 would lose it."""
    _bn_case(lib, C, act, 5, [150, 77, 1, 149], 150, seed=100 + C, utt_offset=3, mean=100.0, std=1e-2)


# ================================================================================================ LayerNorm backward
@pytest.mark.parametrize("M,T,site,utt_offset", [(333, 37, 64, 5), (5000, 250, 69, 0), (4739, 4739, 33, 2), (8, 8, -1, 0), (1, 1, 32, 0)])
def test_ln_bwd(lib, M, T, site, utt_offset):
    from oracle import philox as px
    g = _gen(M + T)
    ypre = torch.randn(M, 512, generator=g, device="cuda") * 2 + 0.5
    dxin = torch.randn(M, 512, generator=g, device="cuda")
    gamma = torch.rand(512, generator=g, device="cuda") + 0.5
    beta = torch.randn(512, generator=g, device="cuda")
    eps, p = 1e-5, 0.1
    thresh = int(p * 4294967296.0)
    dscale = float(torch.tensor(1.0) / torch.tensor(1.0 - p))
    seed_v = 99 + (5 << 32)
    seed_d = _seed_dev(seed_v)
    dy32 = torch.empty(M, 512, device="cuda")
    dsub = torch.empty(M, 512, dtype=torch.bfloat16, device="cuda")
    dg0 = torch.randn(512, generator=g, device="cuda")
    db0 = torch.randn(512, generator=g, device="cuda")
    dg, db = dg0.clone(), db0.clone()
    rc = lib.tts_k_ln_bwd(_p(dxin), _p(ypre), _p(gamma), eps, M, T, _p(dy32), _p(dsub), site, _p(seed_d), utt_offset, thresh, dscale,
                          _p(dg), _p(db), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    y = ypre.to(F64).requires_grad_(True)
    ga = gamma.to(F64).requires_grad_(True)
    be = beta.to(F64).requires_grad_(True)
    out = F.layer_norm(y, (512,), ga, be, eps)
    d = dxin.to(F64)
    out.backward(d)
    xh = (y.detach() - y.detach().mean(1, keepdim=True)) * torch.rsqrt(y.detach().var(1, unbiased=False, keepdim=True) + eps)
    rstd = torch.rsqrt(y.detach().var(1, unbiased=False, keepdim=True) + eps)
    gg = d * ga.detach()
    cond = rstd * (gg.abs() + gg.mean(1, keepdim=True).abs() + (xh * (gg * xh).mean(1, keepdim=True)).abs())
    err = (dy32.to(F64) - y.grad).abs()
    tol = 1e-5 * (y.grad.abs() + cond) + 1e-7
    assert bool((err <= tol).all()), f"dy32: max err / tol {float((err / tol).max()):.3g}"
    assert bool(((dg.to(F64) - dg0.to(F64) - ga.grad).abs() <= 1e-5 * (d * xh).abs().sum(0) + 1e-6).all()), "dgamma"
    assert bool(((db.to(F64) - db0.to(F64) - be.grad).abs() <= 1e-5 * d.abs().sum(0) + 1e-6).all()), "dbeta"
    # dsub16 = bf16(dy * keep * dscale) from the kernel's own dy32: bit for bit, with the oracle's p = 0.1 mask
    if site >= 0:
        m = torch.arange(M)
        keep = px.keep_mask_words(seed_v, site, (m % T).numpy(), (utt_offset + m // T).numpy(), 512, p).cuda()
        want = torch.where(keep > 0, dy32 * dscale, torch.zeros_like(dy32)).to(torch.bfloat16)
    else:
        want = dy32.to(torch.bfloat16)
    assert torch.equal(dsub, want), f"dsub16 differs at {int((dsub != want).sum())} elements"


# ================================================================================================ loss, head gradient
def _loss_case(lib, lens, T, pos_weight, seed, stop_scale=3.0, stop_override=None):
    from oracle.transformer_tts import tts_loss
    B = len(lens)
    g = _gen(seed)
    lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
    before = torch.randn(B, T, 80, generator=g, device="cuda")
    after = torch.randn(B, T, 80, generator=g, device="cuda")
    stop = torch.randn(B, T, generator=g, device="cuda") * stop_scale
    if stop_override is not None:
        stop = stop_override(stop)
    target = torch.randn(B, T, 80, generator=g, device="cuda")
    acc = torch.full((16,), 5.0, device="cuda")
    dbefore = torch.empty(B, T, 80, device="cuda"); dafter = torch.empty_like(dbefore); dstop = torch.empty(B, T, device="cuda")
    loss = torch.empty(1, device="cuda")
    rc = lib.tts_k_loss(_p(before), _p(after), _p(stop), _p(target), _p(lens_t), B, T, pos_weight, _p(acc), _p(dbefore), _p(dafter), _p(dstop),
                        _p(loss), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    xs = [t.cpu().to(F64).requires_grad_(True) for t in (before, after, stop)]
    ref = tts_loss(xs[0], xs[1], xs[2], target.cpu().to(F64), lens_t.cpu(), pos_weight=pos_weight)
    ref.backward()
    # each of the three sums ends in one fp32 accumulator, one atomic add per warp of the loss grid: a rounding of up to
    # half an ulp per add, so the relative error grows with sqrt(adds) (1e-6 for small grids)
    adds = 8 * min((B * T * 81 + 255) // 256, 2368)
    assert abs(float(loss) - ref.item()) <= max(1e-6, EPS32 * adds ** 0.5) * abs(ref.item()), (float(loss), ref.item())
    n = float(sum(lens))
    # dstop: 1 - sigmoid(x) at a large positive logit cancels in fp32, so a few ulps of the gradient's scale (1 + pos_weight) / n
    for name, got, x, atol in (("dbefore", dbefore, xs[0], 1e-9), ("dafter", dafter, xs[1], 1e-9),
                               ("dstop", dstop, xs[2], 4 * EPS32 * (1 + pos_weight) / n)):
        err = (got.cpu().to(F64) - x.grad).abs()
        tol = 1e-5 * x.grad.abs() + atol
        assert bool((err <= tol).all()), f"{name}: max err / tol {float((err / tol).max()):.3g}"
    return before, after, stop, lens_t, dbefore, dafter, dstop


@pytest.mark.parametrize("pos_weight", [5.0, 1.0])
@pytest.mark.parametrize("T,lens", [(37, [37, 20, 1, 36]), (200, [200, 200]), (1, [1]), (800, [800, 1, 333, 799, 512, 64])])
def test_loss(lib, T, lens, pos_weight):
    _loss_case(lib, lens, T, pos_weight, seed=T + len(lens))


@pytest.mark.parametrize("pos_weight", [5.0, 1.0])
def test_loss_saturated_stop_logits(lib, pos_weight):
    """Stop logits of +-40 (both at the positive last frame and elsewhere): softplus must neither overflow nor lose the term."""
    def sat(s):
        return torch.where(s > 0, torch.full_like(s, 40.0), torch.full_like(s, -40.0))
    _loss_case(lib, [50, 1, 23], 50, pos_weight, seed=40, stop_override=sat)


def test_head_grad(lib):
    B, T, lens = 4, 77, [77, 1, 40, 76]
    g = _gen(1)
    lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
    dbefore = torch.randn(B * T, 80, generator=g, device="cuda")
    dafter = torch.randn(B * T, 80, generator=g, device="cuda")
    dpost = torch.randn(B * T, 96, generator=g, device="cuda").to(torch.bfloat16)
    dstop = torch.randn(B * T, generator=g, device="cuda")
    dhead = torch.full((B * T, 128), 9.0, dtype=torch.bfloat16, device="cuda")
    rc = lib.tts_k_head_grad(_p(dbefore), _p(dafter), _p(dpost), 96, _p(dstop), _p(lens_t), B, T, _p(dhead), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    valid = _valid(lens_t, T).reshape(B * T, 1)
    want = torch.zeros(B * T, 128, device="cuda")
    want[:, :80] = (dbefore + dafter + dpost[:, :80].float()) * valid
    want[:, 80] = dstop * valid[:, 0]
    assert torch.equal(dhead, want.to(torch.bfloat16))


# ================================================================================================ word dropout, embedding
@pytest.mark.parametrize("B,T,site,decoder", [(3, 150, 17, 1), (32, 400, 17, 1), (5, 37, 16, 0), (2, 64, -1, 0)])
def test_dropw_bwd(lib, B, T, site, decoder):
    from oracle import philox as px
    g = _gen(B * T)
    M = B * T
    d = torch.randn(M, 512, generator=g, device="cuda")
    pe = torch.randn(T, 512, generator=g, device="cuda")
    p, utt_offset, seed_v = 0.1, 4, 1234567
    thresh = int(p * 4294967296.0)
    dscale = float(torch.tensor(1.0) / torch.tensor(1.0 - p))
    out = torch.empty(M, 512, dtype=torch.bfloat16, device="cuda")
    dalpha = torch.tensor([0.25], device="cuda")
    seed_d = _seed_dev(seed_v)
    rc = lib.tts_k_dropw_bwd(_p(d), _p(out), B, T, site, _p(seed_d), utt_offset, thresh, dscale, _p(pe), _p(dalpha), decoder, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    m = torch.arange(M)
    if site >= 0:
        keep = px.keep_mask_words(seed_v, site, (m % T).numpy(), (utt_offset + m // T).numpy(), 512, p).cuda()
        v32 = torch.where(keep > 0, d * dscale, torch.zeros_like(d))
    else:
        v32 = d
    assert torch.equal(out, v32.to(torch.bfloat16))
    pe_rows = pe[(m % T).cuda()]
    terms = v32.to(F64) * pe_rows.to(F64)
    ref = 0.25 + float(terms.sum())
    assert abs(float(dalpha) - ref) <= 1e-5 * float(terms.abs().sum()), (float(dalpha), ref)


def test_embed_bwd(lib):
    B, S, V = 4, 70, 40
    g = _gen(3)
    lens = torch.tensor([70, 1, 33, 69], dtype=torch.int32, device="cuda")
    ph = torch.randint(0, V + 5, (B, S), generator=g, device="cuda")          # includes the padding id 0 and ids >= V
    ph[0, :10] = 7                                                             # repeated ids accumulate
    d = _ints((B * S, 512), g)
    dE0 = torch.randint(-3, 4, (V, 512), generator=g, device="cuda").float()
    dE = dE0.clone()
    rc = lib.tts_k_embed_bwd(_p(d), _p(ph), _p(lens), B, S, V, _p(dE), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    valid = _valid(lens, S).reshape(-1)
    ids = ph.reshape(-1)
    use = valid & (ids > 0) & (ids < V)
    want = dE0.to(F64).index_add(0, ids[use], d.to(F64)[use])
    assert torch.equal(dE.to(F64), want)
    assert torch.equal(dE[0], dE0[0]), "the padding id gets no gradient"


def test_train_entry_points_reject_bad_arguments(lib):
    assert lib.tts_k_wgrad(None, 8, 8, None, 8, 8, 1, 1, 1, None, None, None) < 0
    assert lib.tts_k_dgrad(None, 8, 8, 5, None, 8, 8, 8, 8, None, None, 8, None, None) < 0
    assert lib.tts_k_bn_train_fwd(None, 1, 1, 6, None, None, None, None, 1e-5, 0, -1, None, 0, None, 8, None, None, None, None) < 0
    assert lib.tts_k_loss(None, None, None, None, None, 1, 1, 5.0, None, None, None, None, None, None) < 0
