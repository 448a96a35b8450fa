"""Cross-attention alignments and FastSpeech durations on a B200 (pytest -m gpu).

Kernel level: tts_k_cross_align against fp64 on the same bf16 inputs.  Integer Q / K with |v| <= 2 make every score an exact
fp32 value, so the argmax is compared bit for bit (engineered ties: first index wins); P and rowmax must fall inside the bound
of the fp32 arithmetic: ex2.approx (relative error <= 2^-22), the rounding of (s - m) * scale_log2, and the fp32 sum of Lk terms.

End to end: tts_forward_align through TransformerTTS.alignments / .durations against the live oracle
(tests/align_reference.py), plus exact self-consistency and invariance checks.
"""
import copy
import ctypes as C
import math

import pytest
import torch

from tests.align_reference import cross_attention_weights, durations_batch
from tests.gpu_util import make_b200_model, rel_l2

pytestmark = pytest.mark.gpu

ULP = 2.0 ** -23


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from transformer_tacotron2_b200 import _lib
    torch.zeros(1, device="cuda")
    return _lib.load()


# ---------------------------------------------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("B,Lq,Lk", [(2, 77, 1), (3, 130, 37), (2, 200, 100), (2, 65, 300), (1, 130, 2048), (4, 33, 64)])
def test_cross_align_kernel_vs_fp64(lib, B, Lq, Lk):
    H = 8
    g = torch.Generator().manual_seed(B * 1000 + Lq + Lk)
    Q = torch.randint(-2, 3, (B, Lq, H * 64), generator=g).float()
    K = torch.randint(-2, 3, (B, H, Lk, 64), generator=g).float()
    Q[:, ::7] = 0                                                     # every valid key ties: argmax must be 0
    if Lk >= 2:
        K[:, :4, 1::2] = K[:, :4, 0:(Lk // 2) * 2:2]                  # heads 0..3: key 2i + 1 = key 2i, the even one must win
    qlens = torch.randint(1, Lq + 1, (B,), generator=g, dtype=torch.int32); qlens[0] = Lq
    klens = torch.randint(1, Lk + 1, (B,), generator=g, dtype=torch.int32); klens[0] = Lk
    if B > 1:
        klens[-1] = 0                                                 # no valid key: zero rows, argmax -1
    Qd, Kd = Q.to(torch.bfloat16).cuda(), K.to(torch.bfloat16).cuda()
    ql, kl = qlens.cuda(), klens.cuda()
    P = torch.full((B, H, Lq, Lk), float("nan"), device="cuda")
    rmax = torch.full((B, H, Lq), float("nan"), device="cuda")
    amax = torch.full((B, H, Lq), 12345, dtype=torch.int16, device="cuda")
    rc = lib.tts_k_cross_align(_p(Qd), H * 64, _p(Kd), _p(ql), _p(kl), B, H, Lq, Lk, _p(P), _p(rmax), _p(amax), _stream())
    assert rc == 0
    # durations-only launch (no P): the same statistics
    rmax2, amax2 = torch.empty_like(rmax), torch.empty_like(amax)
    assert lib.tts_k_cross_align(_p(Qd), H * 64, _p(Kd), _p(ql), _p(kl), B, H, Lq, Lk, None, _p(rmax2), _p(amax2), _stream()) == 0
    torch.cuda.synchronize()
    P, rmax, amax = P.cpu().double(), rmax.cpu().double(), amax.cpu().long()
    assert torch.equal(rmax2.cpu().double(), rmax) and torch.equal(amax2.cpu().long(), amax)

    s = Q.double().view(B, Lq, H, 64).transpose(1, 2) @ K.double().transpose(-1, -2) / 8      # exact (integer / 8)
    kmask = (torch.arange(Lk)[None, :] < klens[:, None])[:, None, None, :]
    qmask = (torch.arange(Lq)[None, :] < qlens[:, None])[:, None, :]
    row_ok = (qmask & (klens > 0)[:, None, None]).expand(B, H, Lq)
    sm = s.masked_fill(~kmask, float("-inf"))
    m = sm.max(-1).values
    ref = torch.softmax(sm, -1).nan_to_num(0.0) * row_ok[..., None]
    want_arg = torch.where(row_ok, sm.argmax(-1), torch.full_like(m, -1, dtype=torch.int64))  # first maximum
    assert torch.equal(amax, want_arg)
    assert (amax[:, :, ::7][row_ok[:, :, ::7]] == 0).all()
    if Lk >= 2:
        assert (amax[:, :4][row_ok[:, :4]] % 2 == 0).all()

    x = ((sm - m[..., None]) * math.log2(math.e)).abs().nan_to_num(0.0, posinf=0.0)         # |exponent| of 2 in the kernel
    kf = klens.double()[:, None, None, None]
    tol = ref * (2e-6 + 2e-7 * x + kf * ULP) + 2e-38
    err = (P - ref).abs()
    print(f"B {B} Lq {Lq} Lk {Lk}: max |dP| {float(err.max()):.3e}, max |dP| / tol {float((err / tol).max()):.3f}")
    assert (err <= tol).all()
    assert (P[~row_ok.unsqueeze(-1).expand_as(P)] == 0).all() and (P[~kmask.expand_as(P)] == 0).all()
    want_max = ref.max(-1).values
    assert ((rmax - want_max).abs() <= want_max * (2e-6 + klens.double()[:, None, None] * ULP)).all()
    assert torch.equal(rmax, P.max(-1).values)                                                # rowmax is the stored maximum
    sums = P.sum(-1)
    lim = (16 + 2 * klens.double())[:, None, None] * ULP
    assert ((sums - 1).abs()[row_ok] <= lim.expand_as(sums)[row_ok]).all(), float((sums - 1).abs()[row_ok].max())


def test_cross_align_argument_errors(lib):
    assert lib.tts_k_cross_align(None, 512, None, None, None, 1, 8, 1, 1, None, None, None, None) < 0
    x = torch.zeros(8, dtype=torch.bfloat16, device="cuda")
    assert lib.tts_k_cross_align(_p(x), 256, _p(x), None, None, 1, 8, 1, 1, None, None, None, None) < 0        # ldq < H * 64


# ---------------------------------------------------------------------------------------------------------------- end to end
B_, S_, T_, SEED_IN = 4, 100, 400, 101
# rel-L2 of P per layer over valid positions against the oracle (bf16 operands, fp32 softmax); measured on a B200:
# 2.0e-3 (layer 0) .. 2.2e-3 (layer 5)
TOL_P = 5e-3


@pytest.fixture(scope="module")
def setup():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from oracle import synthetic
    o = synthetic.make_model(stop_bias=-8.0)
    op = copy.deepcopy(o)                             # planted sharp head: layer 2, head 3 (x 8 on its q and k: bf16-exact)
    with torch.no_grad():
        ca = op.decoder.layers[2].cross_attn
        for lin in (ca.wq, ca.wk):
            lin.weight[3 * 64:4 * 64] *= 8
            lin.bias[3 * 64:4 * 64] *= 8
    inputs = synthetic.make_inputs(B_, S_, T_, SEED_IN, ragged=True)
    return o, make_b200_model(o), op, make_b200_model(op), inputs


def _valid(pl, ml, T, S):
    return ((torch.arange(T)[None, :, None] < ml[:, None, None]) & (torch.arange(S)[None, None, :] < pl[:, None, None]))


def test_alignments_vs_oracle_canonical(setup):
    o, g, _, _, (ph, pl, mels, ml) = setup
    want, _ = cross_attention_weights(o, ph, pl, mels, ml, seed=7)
    got = g.alignments(ph, pl, mels, ml, seed=7)
    assert got.device.type == "cpu" and got.shape == (6, B_, 8, T_, S_)
    v = _valid(pl, ml, T_, S_)[None, :, None].expand_as(got)
    print("canonical: max p", float(want.max()), "F", float(want.max(-1).values.sum(-1).div(ml[None, :, None]).mean()))
    for l in range(6):
        e = rel_l2(got[l][v[l]], want[l][v[l]])
        print(f"layer {l}: P rel-L2 {e:.2e}")
        assert e < TOL_P
    assert (got[~v] == 0).all()


def test_planted_head_durations_vs_oracle(setup):
    _, _, op, g, (ph, pl, mels, ml) = setup
    want, _ = cross_attention_weights(op, ph, pl, mels, ml, seed=7)
    wd, wh, wf = durations_batch(want, pl, ml)
    durs, head, focus = g.durations(ph, pl, mels, ml, seed=7)
    print("planted: oracle F(2,3)", wf[2, :, 3].tolist(), "others max", float(wf[:, :, [0, 1, 2, 4, 5, 6, 7]].max()))
    assert head.tolist() == [19] * B_ and wh.tolist() == [19] * B_
    P = g.alignments(ph, pl, mels, ml, seed=7, layers=[2])[0][:, 3].double()             # [B, T, S]
    ref = want[2][:, 3].double()
    n_ok = n_all = 0
    l1 = 0
    for b in range(B_):
        t, s = int(ml[b]), int(pl[b])
        r, p = ref[b, :t, :s], P[b, :t, :s]
        top2 = r.topk(min(2, s), -1).values
        margin = top2[:, 0] - (top2[:, 1] if s > 1 else 0)
        dp = (p - r).abs().max(-1).values
        ok = margin > 4 * dp
        assert torch.equal(p.argmax(-1)[ok], r.argmax(-1)[ok])
        n_ok += int(ok.sum()); n_all += t
        nq = int((~ok).sum())
        d1 = int((durs[b, :s].long() - wd[b, :s]).abs().sum())
        assert d1 <= 2 * nq, (b, d1, nq)
        l1 += d1
    print(f"planted: {n_ok}/{n_all} frames qualify ({n_ok / n_all:.3f}), |durations - oracle|_1 = {l1}")
    assert n_ok >= 0.8 * n_all
    assert torch.allclose(focus.double()[2, :, 3], wf[2, :, 3], rtol=2e-2)


def test_self_consistency(setup):
    _, _, _, g, (ph, pl, mels, ml) = setup
    phd, pld, md, mld = ph.cuda(), pl.cuda(), mels.cuda(), ml.cuda()
    durs, head, focus = g.durations(phd, pld, md, mld, seed=7)
    assert durs.is_cuda and durs.dtype == torch.int32 and head.dtype == torch.int32
    P = g.alignments(phd, pld, md, mld, seed=7)                                          # [6, B, 8, T, S]
    durs, head, focus, P = durs.cpu(), head.cpu(), focus.cpu(), P.cpu()
    assert durs.sum(1).tolist() == ml.tolist()
    for b in range(B_):
        l, h = divmod(int(head[b]), 8)
        t, s = int(ml[b]), int(pl[b])
        hist = torch.bincount(P[l, b, h, :t, :s].argmax(-1), minlength=S_)
        assert torch.equal(durs[b].long(), hist), b
    want_f = P.max(-1).values.double().sum(-1) / ml.double()[None, :, None]
    assert (focus.double() - want_f).abs().max() < 1e-6
    # durations of a fixed head, and of a layer subset
    d2, h2, f2 = g.durations(ph, pl, mels, ml, seed=7, head=5 * 8 + 6)
    assert h2.tolist() == [46] * B_ and d2.sum(1).tolist() == ml.tolist()
    for b in range(B_):
        hist = torch.bincount(P[5, b, 6, :int(ml[b]), :int(pl[b])].argmax(-1), minlength=S_)
        assert torch.equal(d2[b].long(), hist)
    d3, h3, f3 = g.durations(ph, pl, mels, ml, seed=7, layers=[1, 2])
    assert (f3[[0, 3, 4, 5]] == -1).all() and torch.equal(f3[[1, 2]], focus[[1, 2]])


def test_invariance(setup, lib):
    _, _, _, g, (ph, pl, mels, ml) = setup
    a1 = g.alignments(ph, pl, mels, ml, seed=7)
    a2 = g.alignments(ph, pl, mels, ml, seed=7)
    assert torch.equal(a1, a2)
    d1 = g.durations(ph, pl, mels, ml, seed=7)
    d2 = g.durations(ph, pl, mels, ml, seed=7)
    assert all(torch.equal(x, y) for x, y in zip(d1, d2))
    # a sub-batch starting at utterance 0 (same S, T, utt_offset) reproduces the slice bit for bit
    sub = g.alignments(ph[:2], pl[:2], mels[:2], ml[:2], seed=7)
    assert torch.equal(sub, a1[:, :2])
    ds = g.durations(ph[:2], pl[:2], mels[:2], ml[:2], seed=7)
    assert torch.equal(ds[0], d1[0][:2]) and torch.equal(ds[2], d1[2][:, :2])


def test_forward_align_matches_forward_launch_for_launch(setup, lib):
    _, _, _, g, (ph, pl, mels, ml) = setup
    g.sync_weights()
    hnd, st = g._handle, _stream()
    B, S, T = B_, S_, T_
    ws = g._workspace(B, S, T)
    phd, pld, md, mld = ph.cuda(), pl.cuda().int(), mels.cuda(), ml.cuda().int()
    outs = [torch.empty(B, T, 80, device="cuda"), torch.empty(B, T, 80, device="cuda"), torch.empty(B, T, device="cuda")]
    outs2 = [torch.empty_like(t) for t in outs]
    n0 = lib.tts_launch_count()
    assert lib.tts_forward(hnd, ws.data_ptr(), phd.data_ptr(), pld.data_ptr(), md.data_ptr(), mld.data_ptr(), B, S, T, 7, 0,
                           *[t.data_ptr() for t in outs], st) == 0
    n_fwd = lib.tts_launch_count() - n0
    scratch = torch.empty(lib.tts_align_scratch_bytes(hnd, B, S, T), dtype=torch.uint8, device="cuda")
    P = torch.empty(2, B, 8, T, S, device="cuda")
    focus = torch.empty(6, B, 8, device="cuda")
    durs = torch.empty(B, S, dtype=torch.int32, device="cuda"); head = torch.empty(B, dtype=torch.int32, device="cuda")
    n0 = lib.tts_launch_count()
    rc = lib.tts_forward_align(hnd, ws.data_ptr(), scratch.data_ptr(), phd.data_ptr(), pld.data_ptr(), md.data_ptr(), mld.data_ptr(),
                               B, S, T, 7, 0, 0b100100, -1, *[t.data_ptr() for t in outs2], P.data_ptr(), focus.data_ptr(),
                               durs.data_ptr(), head.data_ptr(), st)
    assert rc == 0, g._lib.tts_last_error_string(hnd)
    n_align = lib.tts_launch_count() - n0
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(outs, outs2))
    assert n_align == n_fwd + 2 + 2                     # two layers' alignment kernels, the focus and the durations kernel
    # heads / postnet skipped when no mel output is wanted
    n0 = lib.tts_launch_count()
    assert lib.tts_forward_align(hnd, ws.data_ptr(), None, phd.data_ptr(), pld.data_ptr(), md.data_ptr(), mld.data_ptr(),
                                 B, S, T, 7, 0, 0b100100, -1, None, None, None, P.data_ptr(), None, None, None, st) == 0
    assert lib.tts_launch_count() - n0 < n_fwd
    # argument checks
    for mask, fixed in ((0, -1), (0x40, -1), (0b100100, 8), (0b100100, 48)):
        assert lib.tts_forward_align(hnd, ws.data_ptr(), scratch.data_ptr(), phd.data_ptr(), pld.data_ptr(), md.data_ptr(),
                                     mld.data_ptr(), B, S, T, 7, 0, mask, fixed, None, None, None, None, None,
                                     durs.data_ptr(), None, st) < 0
    assert lib.tts_forward_align(hnd, ws.data_ptr(), None, phd.data_ptr(), pld.data_ptr(), md.data_ptr(), mld.data_ptr(),
                                 B, S, T, 7, 0, 1, -1, None, None, None, None, None, durs.data_ptr(), None, st) < 0


def test_alignments_of_an_ar_output(setup):
    """inference(return_before=True) then alignments(mel_before): the teacher-forced decoder sees the fed-back frames."""
    _, _, _, g, (ph, pl, mels, ml) = setup
    _, lens, _, mb = g.inference(ph[:2].cuda(), pl[:2].cuda(), max_len=60, seed=7, return_before=True)
    att = g.alignments(ph[:2].cuda(), pl[:2].cuda(), mb, lens, seed=7, layers=[2])
    assert att.shape == (1, 2, 8, mb.shape[1], S_) and att.is_cuda
    sums = att.sum(-1)
    assert torch.allclose(sums, torch.ones_like(sums), atol=1e-4)
    g.train()
    try:
        with pytest.raises(RuntimeError):
            g.durations(ph, pl, mels, ml)
    finally:
        g.eval()
