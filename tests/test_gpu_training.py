"""Training step parity (SURVEY.md 8(a) row a12): train-mode forward, loss, every parameter gradient, BatchNorm running
statistics and one Adam update of the B200 path against the oracle's autograd on the same seeded inputs and the same
Philox dropout masks.  Tolerances (floating point, bf16 operands / fp32 accumulation on the GPU vs fp32 on the CPU) are
written next to each check."""
import copy

import pytest
import torch

from tests.gpu_util import make_b200_model, rel_l2

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="no GPU")]

TOL_OUT = 2e-2        # rel-L2 of train-mode forward outputs
TOL_LOSS = 5e-3       # relative error of the scalar loss
# Gradients: the GPU path differentiates ITS forward (bf16 operands), so ReLU / dropout-gated units whose pre-activation
# is within rounding noise of zero take the other branch than in the fp32 oracle; a flipped fraction f of units costs
# ~sqrt(f) relative L2 on the tensors behind that non-linearity (FFN w1, prenets, convs before BatchNorm+ReLU).
# Measured: 0.4 % (heads) .. 3 % (mid network) .. 7.4 % (encoder prenet convs), whole gradient 1.7-3.6 %.
TOL_GRAD = 1.2e-1     # rel-L2 of every parameter gradient with a non-negligible norm
TOL_GRAD_ALL = 5e-2   # rel-L2 of the whole flat gradient
TOL_GRAD_SCALAR = 1e-1  # enc_alpha / dec_alpha on cases with >= 1000 decoder frames (measured 0.9 % / 2.6 %)


def _check_scalar_grad(name, got, want, n_frames):
    """The alphas' gradients are sums of sign-alternating products over (frames x 512): on tiny cases cancellation turns the
    ~3 % element error into tens of percent of the (small) sum -- and the fp32 atomics make that vary from run to run -- so
    there only sign and order of magnitude are checked; the large cases pin the value."""
    if n_frames >= 1000:
        assert abs(got - want) < TOL_GRAD_SCALAR * abs(want), (name, got, want)
    else:
        assert got * want > 0 and 0.3 < got / want < 3.0, (name, got, want)


def _oracle_step(oracle_model, inputs, seed):
    from oracle.transformer_tts import tts_loss
    ph, pl, mels, ml = inputs
    m = copy.deepcopy(oracle_model).train()
    out = m(ph, pl, mels, ml, seed=seed)
    loss = tts_loss(*out, mels, ml)
    loss.backward()
    return m, [o.detach() for o in out], loss.detach(), {k: p.grad.detach().clone() for k, p in m.named_parameters()}


@pytest.mark.parametrize("B,S,T,ragged", [(3, 12, 20, True), (2, 40, 150, True), (4, 100, 260, False), (1, 7, 13, False), (5, 33, 129, True)])
def test_train_step_gradients(oracle_model, B, S, T, ragged):
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    inputs = synthetic.make_inputs(B, S, T, 900 + B, ragged)
    seed = 7
    om, out_ref, loss_ref, grads_ref = _oracle_step(oracle_model, inputs, seed)

    model = make_b200_model(oracle_model)
    tr = Trainer(model)
    loss = tr.forward_backward(*inputs, seed=seed)
    torch.cuda.synchronize()
    for name, got, want in zip(("mel_before", "mel_after", "stop_logits"), tr.outputs(), out_ref):
        assert rel_l2(got, want) < TOL_OUT, (name, rel_l2(got, want))
    assert abs(float(loss) - float(loss_ref)) / abs(float(loss_ref)) < TOL_LOSS, (float(loss), float(loss_ref))

    grads = tr.grads()
    assert set(grads) == set(grads_ref)
    total_ref = torch.cat([g.flatten() for g in grads_ref.values()]).norm()
    worst = []
    num = 0.0
    for k, want in grads_ref.items():
        got = grads[k]
        assert torch.isfinite(got).all(), k
        num += float((got - want).norm() ** 2)
        if want.norm() > 1e-3 * total_ref:                       # tensors that matter; tiny ones are covered by the global check
            if want.numel() == 1:
                _check_scalar_grad(k, float(got), float(want), B * T)
            else:
                worst.append((rel_l2(got, want), k))
    worst.sort(reverse=True)
    # (BatchNorm statistics over fewer than 16 encoder positions are ill-conditioned: the single-utterance case gets 2x)
    loosen = 2.0 if B * S < 16 else 1.0
    assert worst[0][0] < TOL_GRAD * loosen, worst[:8]
    assert num ** 0.5 / float(total_ref) < TOL_GRAD_ALL * loosen, (num ** 0.5 / float(total_ref), worst[:8])

    # BatchNorm running statistics (P5: momentum 0.1, unbiased variance in the update)
    bufs = tr.buffers()
    for k, v in om.state_dict().items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert torch.allclose(bufs[k], v, atol=2e-2, rtol=2e-2), (k, float((bufs[k] - v).abs().max()))


def test_adam_update_matches_torch(oracle_model):
    """One optimiser step (Vaswani Adam: betas (0.9, 0.98), eps 1e-9): parameters after the step vs torch.optim.Adam fed
    with the gradients the GPU path produced (isolates the optimiser arithmetic from gradient error)."""
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    inputs = synthetic.make_inputs(2, 12, 20, 77, True)
    model = make_b200_model(oracle_model)
    tr = Trainer(model, lr=1e-3)
    tr.forward_backward(*inputs, seed=3)
    grads = tr.grads()
    before = tr.parameters()
    params = {k: torch.nn.Parameter(v.clone()) for k, v in before.items()}
    opt = torch.optim.Adam(list(params.values()), lr=1e-3, betas=(0.9, 0.98), eps=1e-9)
    for k, p in params.items():
        p.grad = grads[k].clone()
    opt.step()
    tr.adam_step()
    after = tr.parameters()
    for k, p in params.items():
        assert torch.allclose(after[k], p.detach(), atol=1e-6, rtol=1e-5), k
    # and the bf16 operand copies were refreshed: a second step runs and the loss moves
    l0 = float(tr._loss)
    l1 = float(tr.forward_backward(*inputs, seed=3))
    assert l1 == l1 and l1 != l0


def test_loss_decreases_over_steps(oracle_model):
    """A few full steps on one fixed batch: the loss goes down (end-to-end sanity of forward + backward + Adam)."""
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    inputs = synthetic.make_inputs(4, 24, 60, 5, True)
    tr = Trainer(make_b200_model(oracle_model), lr=3e-4)
    losses = [float(tr.step(*inputs, seed=100 + i)) for i in range(12)]
    assert all(l == l for l in losses)
    assert min(losses[-3:]) < 0.9 * losses[0], losses        # (a new dropout mask every step: noisy, but clearly down)


def test_data_parallel_shards_match_oracle(oracle_model):
    """Two data-parallel 'ranks' run one after the other on this GPU (utt_offset = first global utterance id of the shard):
    the mean of their flat gradients equals the mean of the oracle's per-shard gradients (per-rank BatchNorm statistics,
    dropout masks keyed by the global utterance id -- SURVEY.md 8(e))."""
    from oracle import synthetic
    from oracle.transformer_tts import tts_loss
    from transformer_tacotron2_b200.training import Trainer
    ph, pl, mels, ml = synthetic.make_inputs(4, 16, 40, 31, True)
    tr = Trainer(make_b200_model(oracle_model))
    got, want = None, None
    for lo, hi in ((0, 2), (2, 4)):
        tr.forward_backward(ph[lo:hi], pl[lo:hi], mels[lo:hi], ml[lo:hi], seed=9, utt_offset=lo)
        g = tr.flat_grads.clone()
        got = g if got is None else got + g
        m = copy.deepcopy(oracle_model).train()
        out = m(ph[lo:hi], pl[lo:hi], mels[lo:hi], ml[lo:hi], seed=9, utt_ids=list(range(lo, hi)))
        tts_loss(*out, mels[lo:hi], ml[lo:hi]).backward()
        ref = {k: p.grad for k, p in m.named_parameters()}
        flat = torch.zeros_like(g, device="cpu")
        for name, off, numel, isb in tr._table:
            if not isb:
                flat[off:off + numel] = ref[name].flatten()
        want = flat if want is None else want + flat
    err = rel_l2(got / 2, want / 2)
    assert err < TOL_GRAD_ALL, err


def test_graph_replay_equals_eager(oracle_model):
    """tts_train_step is replayed from a CUDA graph from the third step of a shape on; with the same inputs and seeds the
    replayed steps produce the loss of the eager steps (atomic accumulation order aside) and honour a NEW seed."""
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    inputs = synthetic.make_inputs(3, 20, 50, 41, True)
    losses = {}
    for mode in (0, 1):
        model = make_b200_model(oracle_model)
        tr = Trainer(model)
        model.set_option("train_graph", mode)
        losses[mode] = [float(tr.forward_backward(*inputs, seed=s)) for s in (1, 1, 1, 2, 1)]
        g = tr.flat_grads.clone()
        losses[mode].append(float(g.norm()))
    eager, graph = losses[0], losses[1]
    assert eager[0] != eager[3]                                        # the seed matters
    for a, b in zip(eager, graph):
        assert abs(a - b) <= 1e-3 * abs(a), (eager, graph)


def test_trained_weights_flow_back_into_inference(oracle_model):
    """Trainer.export_to_module(): after a few optimiser steps the module's state_dict carries the trained parameters and
    BatchNorm statistics; loading that state_dict into the oracle and running the eval-mode forward on both sides agrees
    (the training state and the inference weights are the same numbers)."""
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    inputs = synthetic.make_inputs(3, 16, 40, 8, True)
    model = make_b200_model(oracle_model)
    tr = Trainer(model, lr=2e-4)
    for i in range(3):
        tr.step(*inputs, seed=50 + i)
    tr.export_to_module()
    sd = model.state_dict()
    assert any(not torch.equal(sd[k], v) for k, v in oracle_model.state_dict().items() if v.is_floating_point())
    trained = copy.deepcopy(oracle_model).eval()
    # the kernels read bf16 copies of the matrices; give the oracle the same effective weights so that the comparison
    # measures the flow-back (values, BatchNorm folding of the NEW statistics), not weight quantisation
    trained.load_state_dict({k: (v.to(torch.bfloat16).to(torch.float32) if v.is_floating_point() and v.dim() >= 2 else v) for k, v in sd.items()})
    with torch.no_grad():
        want = trained(*inputs, seed=7)
    got = model(*inputs, seed=7)
    for name, g, w in zip(("mel_before", "mel_after", "stop_logits"), got, want):
        assert rel_l2(g, w) < 2e-2, (name, rel_l2(g, w))


def test_peer_adam_kernel_world1_equals_plain_adam(oracle_model):
    """The fused reduce-scatter -> Adam -> all-gather kernel with a single rank (peers = self) is plain Adam; the multi-GPU
    behaviour is checked by scripts/dp_peer_check.py under torchrun (needs >= 2 GPUs)."""
    import ctypes as C
    from oracle import synthetic
    from transformer_tacotron2_b200.training import Trainer
    inputs = synthetic.make_inputs(2, 12, 20, 3, True)
    ma, mb = make_b200_model(oracle_model), make_b200_model(oracle_model)
    ta, tb = Trainer(ma, lr=1e-3), Trainer(mb, lr=1e-3)
    ta.forward_backward(*inputs, seed=4)
    tb.flat_grads.copy_(ta.flat_grads)          # identical gradients (two backward passes differ in the last bits: atomics)
    ta.adam_step()
    assert tb._lib.tts_train_set_peers(tb._h, 0, 1, None, None) == 0
    mb._check(tb._lib.tts_train_adam_peers(tb._h, 1e-3, 0.9, 0.98, 1e-9, mb._stream()), "adam_peers")
    mb._check(tb._lib.tts_train_repack(tb._h, mb._stream()), "repack")
    pa, pb = ta.parameters(), tb.parameters()
    for k in pa:
        assert torch.allclose(pa[k], pb[k], atol=1e-7, rtol=1e-6), k
    # and the refreshed bf16 operand copies give the same next loss
    la, lb = float(ta.forward_backward(*inputs, seed=5)), float(tb.forward_backward(*inputs, seed=5))
    # (1e-7 parameter differences flip the bf16 rounding of a few weights in the operand copies: allow 2e-3)
    assert abs(la - lb) <= 2e-3 * abs(la), (la, lb)


def test_train_step_vs_committed_golden(oracle_model):
    """The same training step against the committed fixture (tests/golden/train_small.npz, made by make_golden.py from the
    oracle): loss, train-mode outputs, gradient norms of every tensor and the small gradients element-wise."""
    import os
    import numpy as np
    from transformer_tacotron2_b200.training import Trainer
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "train_small.npz"))
    tr = Trainer(make_b200_model(oracle_model))
    loss = tr.forward_backward(torch.from_numpy(g["phonemes"]), torch.from_numpy(g["phoneme_lens"]), torch.from_numpy(g["mels"]),
                               torch.from_numpy(g["mel_lens"]), seed=int(g["seed"]))
    assert abs(float(loss) - float(g["loss"])) < TOL_LOSS * float(g["loss"])
    assert rel_l2(tr.outputs()[1], torch.from_numpy(g["mel_after"])) < TOL_OUT
    grads = tr.grads()
    total = float(np.sqrt((g["grad_norms"] ** 2).sum()))
    for name, want in zip(g["names"], g["grad_norms"]):
        got = float(grads[str(name)].norm())
        if want > 1e-3 * total:
            if grads[str(name)].numel() == 1:                                   # alphas (norm = |value|): see _check_scalar_grad
                assert 0.3 < got / want < 3.0, (str(name), got, float(want))
            else:
                assert abs(got - want) < 0.1 * want, (str(name), got, float(want))
    for key in g.files:
        if key.startswith("grad/"):
            want = torch.from_numpy(g[key])
            if float(want.norm()) > 1e-3 * total and want.numel() > 1:
                assert rel_l2(grads[key[5:]], want) < TOL_GRAD, key
    assert torch.allclose(tr.buffers()["postnet.convs.0.bn.running_mean"], torch.from_numpy(g["bn0_running_mean"]), atol=2e-2, rtol=2e-2)


def test_module_train_mode_forward_autograd(oracle_model):
    """SURVEY.md 8(b): the boundary is the nn.Module -- `model.train(); out = model(...); loss_fn(*out).backward();
    torch.optim.X(model.parameters()).step()` works on the B200 module as on the oracle (autograd bridge over
    tts_train_forward / tts_train_backward), with ANY loss on the outputs."""
    from oracle import synthetic
    from oracle.transformer_tts import tts_loss
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    inputs = synthetic.make_inputs(3, 24, 60, 77, ragged=True)
    ph, pl, mels, ml = inputs
    om, oout, oloss, ograds = _oracle_step(oracle_model, inputs, seed=5)
    g = make_b200_model(oracle_model).train()
    out = g(ph, pl, mels, ml, seed=5)
    assert all(t.requires_grad for t in out)
    for a, b in zip(out, oout):
        assert rel_l2(a, b) < TOL_OUT
    loss = tts_loss(*[t.cpu() for t in out], mels, ml)
    assert abs(float(loss) - float(oloss)) < TOL_LOSS * abs(float(oloss))
    loss.backward()
    num = sum(float((p.grad - ograds[k]).norm() ** 2) for k, p in g.named_parameters()) ** 0.5
    den = sum(float(v.norm() ** 2) for v in ograds.values()) ** 0.5
    print(f"autograd bridge: loss {float(loss):.4f} (oracle {float(oloss):.4f}), whole-gradient rel-L2 {num / den:.4f}")
    assert num / den < TOL_GRAD_ALL
    # BatchNorm running statistics moved exactly as the oracle's
    assert rel_l2(g.postnet.convs[0].bn.running_mean, om.postnet.convs[0].bn.running_mean) < 2e-2
    # a different loss (sum of the stop logits): gradient only behind the stop head path
    g.zero_grad()
    out = g(ph, pl, mels, ml, seed=5)
    out[2].sum().backward()
    assert float(g.stop_linear.weight.grad.norm()) > 0 and float(g.mel_linear.weight.grad.norm()) == 0.0
    # an optimiser step on the module's parameters is picked up by the next forward, and by eval-mode inference
    opt = torch.optim.SGD(g.parameters(), lr=1e-2)
    losses = []
    for _ in range(4):
        opt.zero_grad()
        out = g(ph, pl, mels, ml, seed=5)
        loss = tts_loss(*[t.cpu() for t in out], mels, ml)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    print("autograd bridge losses:", [round(x, 4) for x in losses])
    assert losses[-1] < losses[0]
    g.eval()
    a = g.inference(ph, pl, max_len=8, seed=1)
    assert torch.isfinite(a[0]).all()
