"""CPU: the alignment / duration reference (tests/align_reference.py) the GPU tests compare against."""
import torch

from tests.align_reference import cross_attention_weights, durations_batch, durations_one


def _random_P(L, B, H, T, S, pl, ml, seed, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(L, B, H, T, S, generator=g) * scale
    kmask = torch.arange(S)[None, :] < pl[:, None]
    P = torch.softmax(s.masked_fill(~kmask[None, :, None, None, :], float("-inf")), -1)
    return P * (torch.arange(T)[None, :] < ml[:, None])[None, :, None, :, None]


def test_durations_sum_to_mel_lens():
    pl, ml = torch.tensor([9, 4, 1]), torch.tensor([30, 17, 5])
    P = _random_P(6, 3, 8, 30, 9, pl, ml, 3)
    d, head, focus = durations_batch(P, pl, ml)
    assert d.sum(1).tolist() == ml.tolist()
    for b in range(3):
        assert (d[b, int(pl[b]):] == 0).all()
    assert ((focus > 0) & (focus <= 1)).all()


def test_monotonic_alignment_known_durations():
    want = [3, 1, 4, 2, 5]
    T, S = sum(want), len(want)
    P = torch.full((1, 1, 8, T, S), 1.0 / S)
    rows = torch.repeat_interleave(torch.arange(S), torch.tensor(want))
    P[0, 0, 5] = 0.02
    P[0, 0, 5, torch.arange(T), rows] = 1.0 - 0.02 * (S - 1)        # head 5 is sharp and diagonal
    d, head, _ = durations_batch(P, torch.tensor([S]), torch.tensor([T]))
    assert d[0].tolist() == want and int(head[0]) == 5


def test_ties_go_to_the_first_index():
    P = torch.full((1, 2, 4, 3), 1.0 / 3)                               # [L, H, T, S]: every phoneme and every head ties
    d, focus, idx = durations_one(P)
    assert d.tolist() == [4, 0, 0] and idx == 0
    P = torch.tensor([[[[0.4, 0.1, 0.4, 0.1]]]])
    assert durations_one(P)[0].tolist() == [1, 0, 0, 0]


def test_head_choice_picks_a_planted_sharp_head():
    pl, ml = torch.tensor([20, 12]), torch.tensor([50, 31])
    P = _random_P(6, 2, 8, 50, 20, pl, ml, 5, scale=0.05)              # near-uniform rows everywhere ...
    P[2, :, 3] = _random_P(1, 2, 1, 50, 20, pl, ml, 6, scale=8.0)[0, :, 0]   # ... except layer 2, head 3
    d, head, focus = durations_batch(P, pl, ml)
    assert float(focus[2, :, 3].min()) > 2 * float(focus[:, :, [0, 1, 2, 4, 5, 6, 7]].max())
    assert head.tolist() == [2 * 8 + 3] * 2
    d2, head2, _ = durations_batch(P[[1, 2]], pl, ml, layers=[1, 2])
    assert head2.tolist() == [19, 19] and torch.equal(d2, d)
    d3, head3, _ = durations_batch(P, pl, ml, fixed_head=8 * 4 + 1)
    assert head3.tolist() == [33, 33] and d3.sum(1).tolist() == ml.tolist()


def test_capturing_weights_leaves_forward_bit_identical(oracle_model):
    from oracle import synthetic
    ph, pl, mels, ml = synthetic.make_inputs(2, 12, 20, 17, ragged=True)
    with torch.no_grad():
        want = oracle_model(ph, pl, mels, ml, seed=7)
    P, got = cross_attention_weights(oracle_model, ph, pl, mels, ml, seed=7)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    assert P.shape == (6, 2, 8, 20, 12)
    sums = P.sum(-1)
    valid = (torch.arange(20)[None, :] < ml[:, None])[None, :, None, :].expand_as(sums)
    assert torch.allclose(sums[valid], torch.ones(()), atol=1e-5)
    assert (sums[~valid] == 0).all() and (P[:, 1, :, :, int(pl[1]):] == 0).all()
    with torch.no_grad():                                               # the hooks are gone afterwards
        assert all(torch.equal(a, b) for a, b in zip(oracle_model(ph, pl, mels, ml, seed=7), want))


def test_argument_checks_need_no_gpu():
    import pytest
    from transformer_tacotron2_b200 import TransformerTTS
    assert TransformerTTS._align_layers(None) == (list(range(6)), 0x3F)
    assert TransformerTTS._align_layers([4, 2, 2]) == ([2, 4], 0x14)
    for bad in ([], [6], [-1]):
        with pytest.raises(ValueError):
            TransformerTTS._align_layers(bad)
    m = TransformerTTS().train()
    with pytest.raises(RuntimeError):
        m.alignments(torch.ones(1, 3, dtype=torch.int64), torch.tensor([3]), torch.zeros(1, 4, 80), torch.tensor([4]))
