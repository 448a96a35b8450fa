"""T1: pin the oracle's sub-modules against independent upstream implementations (SURVEY.md 8(c)):
torch.nn.Transformer{Encoder,Decoder}Layer [TT], run live, and torchaudio Tacotron2 [TA], whose outputs on the canonical
weights and the seeded inputs below are stored in tests/golden/upstream_torchaudio.npz (tests/golden/make_upstream_golden.py
regenerates them), so the comparison runs without torchaudio.
The reference repository has no tests or vectors of its own ("parity unpinned" at that boundary)."""
import os

import numpy as np
import torch
import torch.nn as nn

from oracle import synthetic
from oracle.transformer_tts import masked_batchnorm, length_mask, sinusoid_table

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def postnet_input():
    return torch.randn(2, 23, 80, generator=torch.Generator().manual_seed(3))


def encoder_convs_input():
    return torch.randn(2, 512, 19, generator=torch.Generator().manual_seed(4))


def prenet_input():
    return torch.randn(4, 80, generator=torch.Generator().manual_seed(6))


def _torchaudio_outputs(oracle_model):
    g = np.load(os.path.join(GOLD, "upstream_torchaudio.npz"))
    assert str(g["digest"]) == synthetic.state_dict_digest(oracle_model.state_dict())    # stored for these weights
    return g


def _copy_mha(dst: nn.MultiheadAttention, src):
    with torch.no_grad():
        dst.in_proj_weight.copy_(torch.cat([src.wq.weight, src.wk.weight, src.wv.weight]))
        dst.in_proj_bias.copy_(torch.cat([src.wq.bias, src.wk.bias, src.wv.bias]))
        dst.out_proj.weight.copy_(src.wo.weight)
        dst.out_proj.bias.copy_(src.wo.bias)


def _copy(dst, src):
    with torch.no_grad():
        dst.weight.copy_(src.weight)
        dst.bias.copy_(src.bias)


def test_encoder_layer_matches_torch(oracle_model):
    lay = oracle_model.encoder.layers[1]
    ref = nn.TransformerEncoderLayer(512, 8, 2048, dropout=0.0, batch_first=True, norm_first=False).eval()
    _copy_mha(ref.self_attn, lay.self_attn)
    _copy(ref.linear1, lay.ffn.w1); _copy(ref.linear2, lay.ffn.w2)
    _copy(ref.norm1, lay.norm1); _copy(ref.norm2, lay.norm2)
    x = torch.randn(3, 17, 512, generator=torch.Generator().manual_seed(1))
    lens = torch.tensor([17, 9, 13])
    valid = length_mask(lens, 17)
    with torch.no_grad():
        a = lay.self_attn(x, x, valid[:, None, None, :])
        y = lay.norm1(x + a)
        y = lay.norm2(y + lay.ffn(y))
        torch.backends.mha.set_fastpath_enabled(False)
        want = ref(x, src_key_padding_mask=~valid)
    for b in range(3):
        L = int(lens[b])
        assert torch.allclose(y[b, :L], want[b, :L], atol=2e-5, rtol=1e-5)


def test_decoder_layer_matches_torch(oracle_model):
    lay = oracle_model.decoder.layers[2]
    ref = nn.TransformerDecoderLayer(512, 8, 2048, dropout=0.0, batch_first=True, norm_first=False).eval()
    _copy_mha(ref.self_attn, lay.self_attn); _copy_mha(ref.multihead_attn, lay.cross_attn)
    _copy(ref.linear1, lay.ffn.w1); _copy(ref.linear2, lay.ffn.w2)
    _copy(ref.norm1, lay.norm1); _copy(ref.norm2, lay.norm2); _copy(ref.norm3, lay.norm3)
    g = torch.Generator().manual_seed(2)
    x, mem = torch.randn(2, 11, 512, generator=g), torch.randn(2, 7, 512, generator=g)
    tl, sl = torch.tensor([11, 6]), torch.tensor([7, 4])
    tv, sv = length_mask(tl, 11), length_mask(sl, 7)
    causal = torch.tril(torch.ones(11, 11, dtype=torch.bool))
    with torch.no_grad():
        y = lay.norm1(x + lay.self_attn(x, x, causal[None, None] & tv[:, None, None, :]))
        y = lay.norm2(y + lay.cross_attn(y, mem, sv[:, None, None, :]))
        y = lay.norm3(y + lay.ffn(y))
        want = ref(x, mem, tgt_mask=~causal, tgt_key_padding_mask=~tv, memory_key_padding_mask=~sv)
    for b in range(2):
        L = int(tl[b])
        assert torch.allclose(y[b, :L], want[b, :L], atol=2e-5, rtol=1e-5)


def test_postnet_matches_torchaudio_eval(oracle_model):
    x = postnet_input()
    lens = torch.tensor([23, 23])                      # [TA] has no per-layer masking; full lengths
    with torch.no_grad():
        got = oracle_model._postnet(x, lens, 0, np.arange(2))
    want = torch.from_numpy(_torchaudio_outputs(oracle_model)["postnet"])     # [TA] _Postnet(80, 512, 5, 5), eval
    assert torch.allclose(got, want, atol=2e-5, rtol=1e-5)


def test_encoder_convs_match_torchaudio_eval(oracle_model):
    x = encoder_convs_input()
    m = torch.ones(2, 1, 19)
    with torch.no_grad():
        got = x
        for cb in oracle_model.enc_prenet.convs:
            got = torch.relu(masked_batchnorm(cb.bn, cb.conv(got), m, False)) * m
    # [TA] _Encoder(512, 3, 5).convolutions, each followed by ReLU ([TA]:407-408; eval: dropout is identity)
    want = torch.from_numpy(_torchaudio_outputs(oracle_model)["encoder_convs"])
    assert torch.allclose(got, want, atol=2e-5, rtol=1e-5)


def test_masked_batchnorm_training_matches_torch_on_full_lengths():
    bn = nn.BatchNorm1d(6).train(); bn2 = nn.BatchNorm1d(6).train()
    x = torch.randn(3, 6, 10, generator=torch.Generator().manual_seed(5))
    got = masked_batchnorm(bn, x, torch.ones(3, 1, 10), True)
    want = bn2(x)
    assert torch.allclose(got, want, atol=1e-5)
    assert torch.allclose(bn.running_mean, bn2.running_mean, atol=1e-6)
    assert torch.allclose(bn.running_var, bn2.running_var, atol=1e-6)


def test_prenet_matches_torchaudio_structure(oracle_model):
    """[TA] _Prenet: relu(linear) then dropout p=0.5 with training=True even in eval (line 284).
    [TA] has bias=False; with our biases zeroed and masks forced to keep-all the maths coincide."""
    p = oracle_model.dec_prenet
    x = prenet_input()
    out = torch.from_numpy(_torchaudio_outputs(oracle_model)["prenet"])   # [TA] _Prenet with fc1 / fc2 weights, torch.manual_seed(0)
    with torch.no_grad():
        h1 = torch.relu(x @ p.fc1.weight.T)
    # dropout was applied in eval mode: about half of the positive activations are zeroed
    torch.manual_seed(0)
    d1 = torch.nn.functional.dropout(h1, 0.5, training=True)
    want = torch.nn.functional.dropout(torch.relu(d1 @ p.fc2.weight.T), 0.5, training=True)
    assert torch.allclose(out, want, atol=1e-6)
    assert float((d1 == 0).float().mean()) > float((h1 == 0).float().mean()) + 0.1


def test_sinusoid_table_definition():
    pe = sinusoid_table(64, 512)
    assert pe.dtype == torch.float32
    assert torch.allclose(pe[0, 0::2], torch.zeros(256)) and torch.allclose(pe[0, 1::2], torch.ones(256))
    import math
    assert abs(float(pe[5, 10]) - math.sin(5 / 10000 ** (10 / 512))) < 1e-6
    assert abs(float(pe[5, 11]) - math.cos(5 / 10000 ** (10 / 512))) < 1e-6


def test_loss_matches_torch_functional_on_full_lengths():
    """P13: on an unpadded batch the masked-mean loss is F.mse_loss + F.mse_loss + BCEWithLogitsLoss(pos_weight=5) with the
    stop target at the last frame ([TA]-style gate loss; Tacotron 2 sums the before / after MSE terms)."""
    import torch.nn.functional as F
    from oracle.transformer_tts import tts_loss
    g = torch.Generator().manual_seed(5)
    B, T = 3, 17
    mels = torch.randn(B, T, 80, generator=g)
    before, after, stop = torch.randn(B, T, 80, generator=g), torch.randn(B, T, 80, generator=g), torch.randn(B, T, generator=g)
    lens = torch.full((B,), T, dtype=torch.int32)
    target = torch.zeros(B, T); target[:, -1] = 1.0
    want = F.mse_loss(before, mels) + F.mse_loss(after, mels) + \
        F.binary_cross_entropy_with_logits(stop, target, pos_weight=torch.tensor(5.0))
    got = tts_loss(before, after, stop, mels, lens)
    assert torch.allclose(got, want, atol=1e-6, rtol=1e-6)
    # padded frames contribute nothing
    lens2 = torch.tensor([T, T - 5, 3], dtype=torch.int32)
    m = (torch.arange(T)[None, :] < lens2[:, None]).float()
    noisy = tts_loss(before + (1 - m)[..., None] * 100.0, after, stop + (1 - m) * 50.0, mels, lens2)
    clean = tts_loss(before, after, stop, mels, lens2)
    assert torch.allclose(noisy, clean, atol=1e-6)
