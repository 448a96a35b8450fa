"""Multi-speaker synthesis on the B200: the speaker-conditioning kernels against fp64, every path of the module against the live
multi-speaker reference (tests/speaker_reference.py) at the tolerances of test_gpu_parity.py / test_gpu_training.py, invariants
(zero tables = unconditioned model, batch position, sorting, streaming), the staging contract of the C ABI, launch counts, and
training (gradients of the speaker tables, graph replay with new speakers every step, the autograd bridge, export)."""
import copy
import ctypes as C

import pytest
import torch

from tests.gpu_util import make_b200_model, rel_l2
from tests.speaker_reference import SpeakerTTSConfig, make_speaker_model, make_speakers

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="no GPU")]

TOL_MEL, TOL_STOP, TOL_AR, TOL_P = 2e-2, 5e-2, 3e-2, 5e-3
TOL_OUT, TOL_LOSS, TOL_GRAD, TOL_GRAD_ALL = 2e-2, 5e-3, 1.2e-1, 5e-2
CFG = SpeakerTTSConfig(n_speakers=8, spk_embed_dim=16)
STOP_BIAS = -0.505              # tests/golden/inference_small.npz: utterances stop at scattered frames
STOP_CASE_SEED = 338            # B 4, S 30, 48 frames: one utterance stops at frame 40, stop margin 0.077 on the reference


def _gpu(ref, **opts):
    from transformer_tacotron2_b200 import TTSConfig, TransformerTTS
    m = TransformerTTS(TTSConfig(n_speakers=ref.cfg.n_speakers, spk_embed_dim=ref.cfg.spk_embed_dim))
    m.load_state_dict(ref.state_dict())
    for k, v in opts.items():
        m.set_option(k, v)
    return m


@pytest.fixture(scope="module")
def models():
    ref = make_speaker_model(CFG)
    return ref, _gpu(ref)


@pytest.fixture(scope="module")
def lib():
    from transformer_tacotron2_b200 import _lib
    return _lib.load()


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _bf16_ulp(x):
    e = torch.floor(torch.log2(x.abs().clamp(min=1e-30)))
    return torch.pow(2.0, e - 7)


# ------------------------------------------------------------------------------------------------------------- kernels
def test_k_speaker_cond_exact_and_fp64(lib):
    B, NS, D = 6, 5, 40
    g = torch.Generator().manual_seed(1)
    table = torch.randint(-8, 9, (NS, 512), generator=g).float()
    W = torch.randint(-4, 5, (512, D), generator=g).float()
    bias = torch.randint(-4, 5, (512,), generator=g).float()
    sids = torch.tensor([0, 4, 2, 7, -1, 2], dtype=torch.int32)
    js, ks = [3, 0, 39, 7, 5, 11], [1.0, 2.0, 0.25, 7.0, 0.0, 3.0]                 # spembs = k * e_j; k = 0: the zero vector
    spembs = torch.zeros(B, D)
    for b in range(B):
        spembs[b, js[b]] = ks[b]
    dev = [t.cuda() for t in (sids, spembs, table, W, bias)]
    cond, nhat = torch.empty(B, 512, device="cuda"), torch.empty(B, D, device="cuda")
    assert lib.tts_k_speaker_cond(*map(_p, dev[:2]), B, NS, D, *map(_p, dev[2:]), _p(cond), _p(nhat), None) == 0
    torch.cuda.synchronize()
    for b in range(B):
        want = bias.clone()
        if 0 <= int(sids[b]) < NS:
            want += table[int(sids[b])]
        if ks[b] != 0:
            want += W[:, js[b]]
            assert torch.equal(nhat[b].cpu(), torch.nn.functional.one_hot(torch.tensor(js[b]), D).float())
        else:
            assert not nhat[b].cpu().any()
        assert torch.equal(cond[b].cpu(), want), b
    # random values against fp64; and the speaker-ID table alone (no projection)
    sp = torch.randn(B, D, generator=g)
    Wr, br, tr = torch.randn(512, D, generator=g), torch.randn(512, generator=g), torch.randn(NS, 512, generator=g)
    dev = [t.cuda() for t in (sids, sp, tr, Wr, br)]
    assert lib.tts_k_speaker_cond(*map(_p, dev[:2]), B, NS, D, *map(_p, dev[2:]), _p(cond), _p(nhat), None) == 0
    n64 = sp.double() / sp.double().norm(dim=1, keepdim=True)
    want = n64 @ Wr.double().T + br.double()
    ok = (sids >= 0) & (sids < NS)
    want[ok] += tr.double()[sids[ok].long()]
    torch.cuda.synchronize()
    assert (cond.cpu().double() - want).abs().max() < 1e-5 * want.abs().max()
    assert (nhat.cpu().double() - n64).abs().max() < 1e-6
    assert lib.tts_k_speaker_cond(_p(dev[0]), None, B, NS, 0, _p(dev[2]), None, None, _p(cond), None, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(cond[ok.cuda()].cpu(), tr[sids[ok].long()]) and not cond[~ok.cuda()].any()


def test_k_layernorm_cond(lib):
    B, S = 5, 37
    M = B * S
    g = torch.Generator().manual_seed(2)
    x = torch.randn(M, 512, generator=g) * 3 + 1
    gamma, beta = 1 + 0.1 * torch.randn(512, generator=g), 0.1 * torch.randn(512, generator=g)
    xd, gd, bd = x.cuda(), gamma.cuda(), beta.cuda()
    y0, y1 = torch.empty(M, 512, dtype=torch.bfloat16, device="cuda"), torch.empty(M, 512, dtype=torch.bfloat16, device="cuda")
    zero = torch.zeros(B, 512, device="cuda")
    assert lib.tts_k_layernorm(_p(xd), _p(gd), _p(bd), _p(y0), M, C.c_float(1e-5), None) == 0
    assert lib.tts_k_layernorm_cond(_p(xd), _p(gd), _p(bd), _p(zero), _p(y1), M, S, C.c_float(1e-5), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(y0.view(torch.int16), y1.view(torch.int16))
    cond = torch.randn(B, 512, generator=g)
    cd = cond.cuda()
    assert lib.tts_k_layernorm_cond(_p(xd), _p(gd), _p(bd), _p(cd), _p(y1), M, S, C.c_float(1e-5), None) == 0
    x64 = x.double()
    ln = (x64 - x64.mean(1, keepdim=True)) / torch.sqrt(x64.var(1, unbiased=False, keepdim=True) + 1e-5)
    terms = (ln * gamma.double(), beta.double().expand(M, 512), cond.double().repeat_interleave(S, 0))
    want = terms[0] + terms[1] + terms[2]
    torch.cuda.synchronize()
    # one bf16 ulp of the result, plus the fp32 rounding of the terms summed before it (visible where they cancel)
    bound = _bf16_ulp(want) + 2.0 ** -20 * sum(t.abs() for t in terms)
    err = (y1.cpu().double() - want).abs()
    assert bool((err <= bound).all()), float((err / bound).max())


def test_k_speaker_cond_bwd_exact_and_repeatable(lib):
    B, S, NS, D = 5, 7, 4, 24
    g = torch.Generator().manual_seed(3)
    plens = torch.tensor([7, 3, 1, 5, 2], dtype=torch.int32)
    sids = torch.tensor([1, 3, 1, 0, 3], dtype=torch.int32)                # duplicates; speaker 2 unused
    dmem = torch.randint(-3, 4, (B * S, 512), generator=g).float()
    for b in range(B):
        dmem[b * S + int(plens[b]):(b + 1) * S] = 1000.0                     # rows past plens must not count
    nhat = torch.randint(-2, 3, (B, D), generator=g).float()
    dcond_w = torch.stack([dmem[b * S:b * S + int(plens[b])].sum(0) for b in range(B)])
    dE_w = torch.full((NS, 512), 0.5)
    for b in range(B):
        dE_w[int(sids[b])] += dcond_w[b]
    dW_w, db_w = 0.25 + dcond_w.T @ nhat, -1 + dcond_w.sum(0)

    def run(dm, nh):
        out = [torch.empty(B, 512, device="cuda"), torch.full((NS, 512), 0.5, device="cuda"), torch.full((512, D), 0.25, device="cuda"),
               torch.full((512,), -1.0, device="cuda")]
        args = [t.cuda() for t in (dm, plens, sids, nh)]                     # (kept alive until the kernel has run)
        assert lib.tts_k_speaker_cond_bwd(*map(_p, args), B, S, NS, D, *map(_p, out), None) == 0
        torch.cuda.synchronize()
        return [t.cpu() for t in out]

    dcond, dE, dW, db = run(dmem, nhat)
    assert torch.equal(dcond, dcond_w) and torch.equal(dE, dE_w) and torch.equal(dW, dW_w) and torch.equal(db, db_w)
    assert (dE[2] == 0.5).all()                                              # the unused speaker's row is untouched
    dm, nh = torch.randn(B * S, 512, generator=g), torch.randn(B, D, generator=g)
    a, b_ = run(dm, nh), run(dm, nh)
    assert all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(a, b_))


# ------------------------------------------------------------------------------------------------------------- end to end
def _batch(B, S, T, seed):
    from oracle import synthetic
    ph, pl, mels, ml = synthetic.make_inputs(B, S, T, seed, ragged=True)
    sids, spembs = make_speakers(B, CFG, seed)
    return ph, pl, mels, ml, sids, spembs


def test_encode_vs_reference(models):
    ref, g = models
    ph, pl, _, _, sids, spembs = _batch(3, 50, 8, 31)
    with torch.no_grad():
        want = ref.encode(ph, pl, sids=sids, spembs=spembs)
    got = g.encode(ph, pl, sids=sids, spembs=spembs).cpu()
    for b in range(3):
        L = int(pl[b])
        assert rel_l2(got[b, :L], want[b, :L]) < TOL_MEL


@pytest.mark.parametrize("B,S,T,seed", [(2, 12, 20, 201), (3, 37, 129, 33)])
def test_forward_vs_reference(models, B, S, T, seed):
    ref, g = models
    ph, pl, mels, ml, sids, spembs = _batch(B, S, T, seed)
    with torch.no_grad():
        mb, ma, st = ref(ph, pl, mels, ml, seed=7, sids=sids, spembs=spembs)
    gb, ga, gs = (t.cpu() for t in g(ph, pl, mels, ml, seed=7, sids=sids, spembs=spembs))
    print("forward rel-L2", rel_l2(gb, mb), rel_l2(ga, ma), "stop max-abs", float((gs - st).abs().max()))
    assert rel_l2(gb, mb) < TOL_MEL and rel_l2(ga, ma) < TOL_MEL
    assert float((gs - st).abs().max()) < TOL_STOP


def test_alignments_vs_reference(models):
    from tests.align_reference import cross_attention_weights
    ref, g = models
    B, S, T = 3, 21, 40
    ph, pl, mels, ml, sids, spembs = _batch(B, S, T, 55)

    class Bound:                                   # the reference with this batch's speakers bound, as the hooks expect a model
        decoder = ref.decoder

        def __call__(self, *a, **k):
            return ref(*a, sids=sids, spembs=spembs, **k)

    want, _ = cross_attention_weights(Bound(), ph, pl, mels, ml, seed=7)
    got = g.alignments(ph, pl, mels, ml, seed=7, sids=sids, spembs=spembs)
    v = ((torch.arange(T)[None, :, None] < ml[:, None, None]) & (torch.arange(S)[None, None, :] < pl[:, None, None]))[:, None]
    v = v.expand(B, 8, T, S)
    for l in range(6):
        assert rel_l2(got[l][v], want[l][v]) < TOL_P, l
    durs, head, _ = g.durations(ph, pl, mels, ml, seed=7, sids=sids, spembs=spembs)
    assert durs.sum(1).tolist() == ml.tolist()


def test_inference_stop_case_vs_reference():
    from oracle import synthetic
    ref = make_speaker_model(CFG, stop_bias=STOP_BIAS)
    g = _gpu(ref)
    ph, pl, _, _ = synthetic.make_inputs(4, 30, 8, STOP_CASE_SEED, ragged=True)
    sids, spembs = make_speakers(4, CFG, STOP_CASE_SEED)
    ma, lens, st = ref.inference(ph, pl, max_len=48, seed=7, sids=sids, spembs=spembs)
    ga, gl, gs = (t.cpu() for t in g.inference(ph.cuda(), pl.cuda(), max_len=48, seed=7, sids=sids.cuda(), spembs=spembs.cuda()))
    T = min(ga.shape[1], ma.shape[1])
    valid = torch.arange(T)[None, :] < torch.minimum(lens, gl)[:, None]
    err = float(((gs[:, :T] - st[:, :T]).abs() * valid).max())
    margin = float(st[:, :T].abs()[valid].min())
    print(f"AR: lens {lens.tolist()} gpu {gl.tolist()} stop err {err:.4f} margin {margin:.4f} rel-L2 {rel_l2(ga[:, :T], ma[:, :T]):.4f}")
    assert min(lens.tolist()) < 48 and err < TOL_STOP and margin > 4 * err
    assert gl.tolist() == lens.tolist()
    assert ga.shape == ma.shape and rel_l2(ga, ma) < TOL_AR
    # CPU inputs of a conditioned model take the device path and give the same result
    ca, cl, cs = g.inference(ph, pl, max_len=48, seed=7, sids=sids, spembs=spembs)
    assert torch.equal(ca, ga) and torch.equal(cl, gl) and torch.equal(cs, gs)


# ------------------------------------------------------------------------------------------------------------- invariants
def test_zero_tables_bit_identical_to_unconditioned():
    from oracle import synthetic
    z = _gpu(make_speaker_model(CFG, stop_bias=STOP_BIAS, zero=True))
    u = make_b200_model(synthetic.make_model(stop_bias=STOP_BIAS))
    ph, pl, mels, ml, sids, spembs = _batch(5, 24, 30, 12)
    spk = dict(sids=sids, spembs=spembs)
    for a, b in zip(z(ph, pl, mels, ml, seed=3, **spk), u(ph, pl, mels, ml, seed=3)):
        assert torch.equal(a, b)
    phd, pld = ph.cuda(), pl.cuda()
    ia, ib = z.inference(phd, pld, max_len=40, seed=3, **spk), u.inference(phd, pld, max_len=40, seed=3)
    assert all(torch.equal(a, b) for a, b in zip(ia, ib))
    ca = [c.mel_after for c in z.inference_stream(phd, pld, max_len=40, seed=3, chunk_frames=16, **spk)]
    cb = [c.mel_after for c in u.inference_stream(phd, pld, max_len=40, seed=3, chunk_frames=16)]
    assert torch.equal(torch.cat(ca, 1), torch.cat(cb, 1))
    for a, b in zip(z.durations(ph, pl, mels, ml, seed=3, **spk), u.durations(ph, pl, mels, ml, seed=3)):
        assert torch.equal(a, b)


def test_speakers_matter_and_batch_position_does_not(models):
    _, g = models
    ph, pl, _, _, sids, spembs = _batch(6, 20, 8, 77)
    phd, pld = ph.cuda(), pl.cuda()
    a = g.inference(phd, pld, max_len=30, seed=5, sids=sids, spembs=spembs)
    other = (sids + 1) % CFG.n_speakers
    b = g.inference(phd, pld, max_len=30, seed=5, sids=other, spembs=spembs)
    for i in range(6):
        assert not torch.equal(a[0][i], b[0][i])
    # the same utterance, id and speaker at another batch position: bit-identical
    perm = torch.tensor([3, 0, 5, 1, 4, 2])
    c = g.inference(phd[perm.cuda()], pld[perm.cuda()], max_len=30, seed=5, utt_ids=perm.tolist(), sids=sids[perm], spembs=spembs[perm])
    T = c[0].shape[1]
    assert torch.equal(c[0], a[0][perm.cuda(), :T]) and torch.equal(c[1], a[1][perm.cuda()])
    # sorted decoding returns the caller's order, bit for bit
    s = g.inference(phd, pld, max_len=30, seed=5, sids=sids, spembs=spembs, sort_by_length=True, max_lens=[30, 9, 17, 30, 4, 22])
    r = g.inference(phd, pld, max_len=30, seed=5, sids=sids, spembs=spembs, max_lens=[30, 9, 17, 30, 4, 22])
    assert all(torch.equal(x, y) for x, y in zip(s, r))


def test_stream_chunks_concatenate_to_inference(models):
    _, g = models
    ph, pl, _, _, sids, spembs = _batch(5, 18, 8, 91)
    phd, pld = ph.cuda(), pl.cuda()
    ma, ml, st = g.inference(phd, pld, max_len=45, seed=2, sids=sids, spembs=spembs)
    chunks = list(g.inference_stream(phd, pld, max_len=45, seed=2, chunk_frames=12, sids=sids, spembs=spembs))
    assert torch.equal(torch.cat([c.mel_after for c in chunks], 1), ma)
    assert torch.equal(torch.cat([c.stop_logits for c in chunks], 1), st)
    assert torch.equal(sum(c.n_valid for c in chunks), ml)


def test_staging_contract(models, lib):
    ref, g = models
    ph, pl, _, _, sids, spembs = _batch(2, 10, 8, 5)
    g.encode(ph, pl, sids=sids, spembs=spembs)                               # handle and weights ready
    h, ws, st = g._handle, g._workspace(2, 10, 10), g._stream()
    phd, pld = ph.cuda(), pl.cuda().int()
    sd, sp = sids.cuda().int(), spembs.cuda()
    E_STATE = -2
    assert lib.tts_encode(h, _p(ws), _p(phd), _p(pld), 2, 10, 10, None, st) == E_STATE       # nothing staged
    assert lib.tts_set_conditioning(h, _p(ws), 2, _p(sd), None, st) != 0                     # spembs missing
    assert lib.tts_set_conditioning(h, _p(ws), 2, _p(sd), _p(sp), st) == 0
    assert lib.tts_encode(h, _p(ws), _p(phd), _p(pld), 1, 10, 10, None, st) == E_STATE       # staged for another B
    assert lib.tts_set_conditioning(h, _p(ws), 2, _p(sd), _p(sp), st) == 0
    assert lib.tts_encode(h, _p(ws), _p(phd), _p(pld), 2, 10, 10, None, st) == 0
    assert lib.tts_encode(h, _p(ws), _p(phd), _p(pld), 2, 10, 10, None, st) == E_STATE       # consumed
    ma, st_h, ml_h, pl_h = torch.empty(2, 8, 80), torch.empty(2, 8), torch.empty(2, dtype=torch.int32), pl.int()
    tout = C.c_int(0)
    assert lib.tts_infer_host(h, _p(ws), _p(ph), _p(pl_h), 2, 10, 8, 7, 0, _p(ma), _p(ml_h), _p(st_h), C.byref(tout), st) == E_STATE
    for bad in (dict(sids=torch.tensor([0, CFG.n_speakers])), dict(sids=torch.tensor([0, -1])), dict(sids=None)):
        with pytest.raises(ValueError):
            g.inference(phd, pld, max_len=8, **{"sids": sids, "spembs": spembs, **bad})
    from oracle import synthetic
    u = make_b200_model(synthetic.make_model())
    u.encode(ph, pl)
    assert lib.tts_set_conditioning(u._handle, _p(u._workspace(2, 10, 10)), 2, _p(sd), _p(sp), u._stream()) == E_STATE
    with pytest.raises(ValueError):
        u.encode(ph, pl, sids=sids)


def test_launch_counts(models, lib):
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    ref, g = models
    u = make_b200_model(synthetic.make_model())
    ph, pl, mels, ml, sids, spembs = _batch(3, 16, 24, 6)
    counts = []
    for m, spk in ((u, {}), (g, dict(sids=sids, spembs=spembs))):
        m.encode(ph, pl, **spk)
        torch.cuda.synchronize()
        n0 = lib.tts_launch_count()
        m.encode(ph, pl, **spk)
        counts.append(lib.tts_launch_count() - n0)
    assert counts[1] == counts[0] + 1, counts                                   # the speaker-vector kernel; LayerNorm is fused
    steps = []
    for m, spk in ((u, {}), (_gpu(ref), dict(sids=sids, spembs=spembs))):
        m.set_option("train_graph", 0)
        tr = Trainer(m)
        tr.forward_backward(ph, pl, mels, ml, seed=1, **spk)
        n0 = lib.tts_launch_count()
        tr.forward_backward(ph, pl, mels, ml, seed=1, **spk)
        steps.append(lib.tts_launch_count() - n0)
    assert steps[1] == steps[0] + 3, steps                                      # speaker vector, dcond, parameter gradients


# ------------------------------------------------------------------------------------------------------------- training
def _reference_step(ref, inputs, spk, seed):
    from oracle.transformer_tts import tts_loss
    ph, pl, mels, ml = inputs
    m = copy.deepcopy(ref).train()
    out = m(ph, pl, mels, ml, seed=seed, **spk)
    loss = tts_loss(*out, mels, ml)
    loss.backward()
    return m, [o.detach() for o in out], loss.detach(), {k: p.grad.detach().clone() for k, p in m.named_parameters()}


@pytest.mark.parametrize("B,S,T", [(3, 12, 20), (4, 40, 150)])
def test_train_gradients_vs_reference(models, B, S, T):
    from transformer_tacotron2_b200.training import Trainer
    ref, _ = models
    ph, pl, mels, ml, sids, spembs = _batch(B, S, T, 900 + B)
    spk = dict(sids=sids, spembs=spembs)
    _, out_ref, loss_ref, grads_ref = _reference_step(ref, (ph, pl, mels, ml), spk, 7)
    tr = Trainer(_gpu(ref))
    loss = tr.forward_backward(ph, pl, mels, ml, seed=7, **spk)
    for got, want in zip(tr.outputs(), out_ref):
        assert rel_l2(got, want) < TOL_OUT
    assert abs(float(loss) - float(loss_ref)) < TOL_LOSS * abs(float(loss_ref))
    grads = tr.grads()
    assert set(grads) == set(grads_ref)
    total = torch.cat([v.flatten() for v in grads_ref.values()]).norm()
    num, worst = 0.0, []
    for k, want in grads_ref.items():
        num += float((grads[k] - want).norm() ** 2)
        if want.numel() > 1 and want.norm() > 1e-3 * total:
            worst.append((rel_l2(grads[k], want), k))
    worst.sort(reverse=True)
    print("worst", worst[:4], "speaker", [(k, e) for e, k in worst if k.startswith(("speaker_embed", "spk_proj"))])
    assert worst[0][0] < TOL_GRAD, worst[:8]
    assert num ** 0.5 / float(total) < TOL_GRAD_ALL
    for k in ("speaker_embed.weight", "spk_proj.weight", "spk_proj.bias"):
        assert rel_l2(grads[k], grads_ref[k]) < TOL_GRAD, k
    unused = sorted(set(range(CFG.n_speakers)) - set(sids.tolist()))
    assert unused and not grads["speaker_embed.weight"][unused].any()


def test_graph_replay_with_new_speakers_every_step(models):
    """Steps replayed from the captured graph read each step's newly staged speakers: exactly the rows of that step's speakers get
    a gradient, and the same sequence of batches gives the losses and speaker-table gradients of the eager steps.  (Two runs of
    the step differ in the last bits -- atomics elsewhere in the step -- and the table gradient, a sum over every memory row,
    amplifies that: 0.6 % rel-L2 was measured between an eager and a replayed run; the tolerance is 2 %.)"""
    from transformer_tacotron2_b200.training import Trainer
    ref, _ = models
    ph, pl, mels, ml, _, spembs = _batch(3, 20, 50, 41)
    plan = [torch.tensor([0, 1, 2]), torch.tensor([3, 3, 5]), torch.tensor([7, 0, 6]), torch.tensor([2, 2, 2])]
    res = {}
    for mode in (0, 1):
        m = _gpu(ref, train_graph=mode)
        tr = Trainer(m)
        res[mode] = []
        for s in plan:
            loss = float(tr.forward_backward(ph, pl, mels, ml, seed=1, sids=s, spembs=spembs))
            gE = tr.grads()["speaker_embed.weight"]
            assert set(torch.nonzero(gE.abs().sum(1)).flatten().tolist()) == set(s.tolist()), (mode, s)
            res[mode].append((loss, gE))
    for (le, ge), (lg, gg) in zip(res[0], res[1]):
        assert abs(le - lg) <= 1e-3 * abs(le)
        assert rel_l2(gg, ge) < 2e-2
    assert len({round(r[0], 6) for r in res[1]}) == len(plan)                 # every replay saw its own speakers


def test_autograd_bridge_and_export(models):
    from oracle.transformer_tts import tts_loss
    from transformer_tacotron2_b200.training import Trainer
    ref, _ = models
    ph, pl, mels, ml, sids, spembs = _batch(3, 24, 60, 77)
    spk = dict(sids=sids, spembs=spembs)
    _, _, oloss, ograds = _reference_step(ref, (ph, pl, mels, ml), spk, 5)
    g = _gpu(ref).train()
    out = g(ph, pl, mels, ml, seed=5, **spk)
    loss = tts_loss(*[t.cpu() for t in out], mels, ml)
    assert abs(float(loss.detach()) - float(oloss)) < TOL_LOSS * abs(float(oloss))
    loss.backward()
    assert rel_l2(g.speaker_embed.weight.grad, ograds["speaker_embed.weight"]) < TOL_GRAD
    assert rel_l2(g.spk_proj.weight.grad, ograds["spk_proj.weight"]) < TOL_GRAD
    # Trainer steps move the speaker table; after export, inference uses the trained table
    m = _gpu(ref)
    before = m.speaker_embed.weight.detach().clone()
    tr = Trainer(m, lr=1e-3)
    for i in range(3):
        tr.step(ph, pl, mels, ml, seed=10 + i, **spk)
    tr.export_to_module()
    assert not torch.equal(m.speaker_embed.weight, before)
    fresh = _gpu(ref)
    fresh.load_state_dict(m.state_dict())
    phd, pld = ph.cuda(), pl.cuda()
    a = m.eval().inference(phd, pld, max_len=20, seed=3, **spk)
    b = fresh.inference(phd, pld, max_len=20, seed=3, **spk)
    c = _gpu(ref).inference(phd, pld, max_len=20, seed=3, **spk)
    assert torch.equal(a[0], b[0]) and not torch.equal(a[0], c[0])
