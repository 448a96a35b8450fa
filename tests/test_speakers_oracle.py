"""CPU: the multi-speaker reference (tests/speaker_reference.py) and the module's speaker parameters and argument checks."""
import pytest
import torch
import torch.nn.functional as F

from oracle import synthetic
from tests.speaker_reference import SpeakerTTSConfig, make_speaker_model, make_speakers

CFG = SpeakerTTSConfig(n_speakers=7, spk_embed_dim=24)


def test_default_config_keys_and_weights_unchanged():
    from transformer_tacotron2_b200 import TTSConfig as ProductConfig, TransformerTTS
    base = synthetic.make_model()
    assert list(TransformerTTS().state_dict()) == list(base.state_dict())
    assert ProductConfig().n_speakers == 0 and ProductConfig().spk_embed_dim == 0
    # the reference with no speakers is the oracle, weight for weight
    m = make_speaker_model(SpeakerTTSConfig())
    assert synthetic.state_dict_digest(m.state_dict()) == synthetic.state_dict_digest(base.state_dict())


def test_speaker_parameters_come_last_and_keep_the_seeded_base():
    from transformer_tacotron2_b200 import TTSConfig as ProductConfig, TransformerTTS
    torch.manual_seed(3)
    a = TransformerTTS()
    torch.manual_seed(3)
    b = TransformerTTS(ProductConfig(n_speakers=5, spk_embed_dim=16))
    ka, kb = list(a.state_dict()), list(b.state_dict())
    assert kb[:len(ka)] == ka and kb[len(ka):] == ["speaker_embed.weight", "spk_proj.weight", "spk_proj.bias"]
    for k in ka:
        assert torch.equal(a.state_dict()[k], b.state_dict()[k]), k
    assert b.speaker_embed.weight.shape == (5, 512) and b.spk_proj.weight.shape == (512, 16)
    assert b.speaker_embed.padding_idx is None
    # the reference carries the same keys as the product module
    ref = make_speaker_model(SpeakerTTSConfig(n_speakers=5, spk_embed_dim=16))
    assert list(ref.state_dict()) == kb
    base = synthetic.make_model()
    for k, v in base.state_dict().items():
        assert torch.equal(ref.state_dict()[k], v), k


def test_zero_tables_equal_unconditioned_oracle():
    ph, pl, mels, ml = synthetic.make_inputs(3, 14, 12, 5, ragged=True)
    sids, spembs = make_speakers(3, CFG, 1)
    o = synthetic.make_model(stop_bias=-0.45)
    z = make_speaker_model(CFG, stop_bias=-0.45, zero=True)
    with torch.no_grad():
        for a, b in zip(o(ph, pl, mels, ml, seed=7), z(ph, pl, mels, ml, seed=7, sids=sids, spembs=spembs)):
            assert torch.equal(a, b)
        for a, b in zip(o.inference(ph, pl, max_len=10, seed=7), z.inference(ph, pl, max_len=10, seed=7, sids=sids, spembs=spembs)):
            assert torch.equal(a, b)


def test_memory_is_encoder_output_plus_speaker_vector():
    ph, pl, _, _ = synthetic.make_inputs(4, 9, 4, 8, ragged=True)
    sids, spembs = make_speakers(4, CFG, 2)
    m = make_speaker_model(CFG)
    o = synthetic.make_model()
    with torch.no_grad():
        hs = o.encode(ph, pl)
        want = hs + m.speaker_embed.weight[sids][:, None, :] + F.linear(spembs / spembs.norm(dim=1, keepdim=True).clamp(min=1e-12),
                                                                        m.spk_proj.weight, m.spk_proj.bias)[:, None, :]
        got = m.encode(ph, pl, sids=sids, spembs=spembs)
    assert torch.allclose(got, want, atol=1e-5, rtol=1e-5)
    # every row, padded ones included, carries the speaker vector
    assert not torch.allclose(got[:, -1], hs[:, -1])


def test_reference_argument_checks():
    ph, pl, mels, ml = synthetic.make_inputs(2, 6, 5, 9, ragged=False)
    sids, spembs = make_speakers(2, CFG, 3)
    m = make_speaker_model(CFG)
    with pytest.raises(ValueError):
        m(ph, pl, mels, ml, sids=sids)                                   # spembs missing
    with pytest.raises(ValueError):
        make_speaker_model(SpeakerTTSConfig()).encode(ph, pl, sids=sids)  # unconditioned model


def test_spembs_get_no_gradient_and_tables_do():
    ph, pl, mels, ml = synthetic.make_inputs(2, 6, 5, 9, ragged=True)
    sids, spembs = make_speakers(2, CFG, 3)
    spembs = spembs.clone().requires_grad_(True)
    m = make_speaker_model(CFG).train()
    out = m(ph, pl, mels, ml, seed=1, sids=sids, spembs=spembs)
    sum(o.sum() for o in out).backward()
    assert spembs.grad is None
    g = m.speaker_embed.weight.grad
    used = set(sids.tolist())
    for j in range(CFG.n_speakers):
        assert (float(g[j].abs().sum()) > 0) == (j in used)
    assert float(m.spk_proj.weight.grad.norm()) > 0


def test_module_validates_speaker_inputs_on_the_host():
    from transformer_tacotron2_b200 import TTSConfig as ProductConfig, TransformerTTS
    m = TransformerTTS(ProductConfig(n_speakers=4, spk_embed_dim=8))
    ok = (torch.tensor([0, 3]), torch.randn(2, 8))
    for sids, spembs in [(None, ok[1]), (ok[0], None), (torch.tensor([0, 4]), ok[1]), (torch.tensor([-1, 0]), ok[1]),
                         (torch.tensor([0.0, 1.0]), ok[1]), (torch.tensor([0, 1, 2]), ok[1]), (ok[0], torch.randn(2, 7)),
                         (ok[0], torch.ones(2, 8, dtype=torch.int64))]:
        with pytest.raises(ValueError):
            m._speaker_inputs(sids, spembs, 2)
    with pytest.raises(ValueError):
        TransformerTTS()._speaker_inputs(ok[0], None, 2)
    assert TransformerTTS()._speaker_inputs(None, None, 2) is None
