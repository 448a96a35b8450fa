"""CPU: import / export of multi-speaker ESPnet Transformer-TTS checkpoints (sid_emb, x-vector projection), synthetic state dicts."""
import pytest
import torch

from transformer_tacotron2_b200 import TTSConfig, TransformerTTS
from transformer_tacotron2_b200 import interchange as ic


@pytest.fixture(scope="module")
def ref_sd():
    torch.manual_seed(0)
    return TransformerTTS(TTSConfig(n_speakers=6, spk_embed_dim=32)).state_dict()


def test_multi_speaker_round_trip(ref_sd):
    esp = ic.to_espnet_state_dict(ref_sd)
    assert torch.equal(esp["sid_emb.weight"], ref_sd["speaker_embed.weight"])
    assert torch.equal(esp["projection.weight"], ref_sd["spk_proj.weight"]) and torch.equal(esp["projection.bias"], ref_sd["spk_proj.bias"])
    assert "encoder.embed.0.projection.weight" in esp                     # the prenet projection keeps its own name
    back = ic.from_espnet_state_dict({"tts." + k: v for k, v in esp.items()}, ref_sd, spk_embed_integration_type="add")
    assert set(back) == set(ref_sd)
    for k, v in ref_sd.items():
        assert torch.equal(back[k].to(v.dtype), v), k


def test_speaker_id_only_needs_no_integration_type():
    torch.manual_seed(0)
    sd = TransformerTTS(TTSConfig(n_speakers=4)).state_dict()
    back = ic.from_espnet_state_dict(ic.to_espnet_state_dict(sd), sd)
    assert torch.equal(back["speaker_embed.weight"], sd["speaker_embed.weight"])


def test_refusals(ref_sd):
    esp = ic.to_espnet_state_dict(ref_sd)
    with pytest.raises(ic.InterchangeError, match="spk_embed_integration_type"):
        ic.from_espnet_state_dict(esp, ref_sd)                                             # projection without the type
    with pytest.raises(ic.InterchangeError, match="concat"):
        ic.from_espnet_state_dict(esp, ref_sd, spk_embed_integration_type="concat")
    with pytest.raises(ic.InterchangeError, match="lid_emb"):
        ic.from_espnet_state_dict({**esp, "lid_emb.weight": torch.zeros(3, 512)}, ref_sd, spk_embed_integration_type="add")
    with pytest.raises(ic.InterchangeError, match="gst"):
        ic.from_espnet_state_dict({**esp, "gst.stl.gst_embs": torch.zeros(10, 256)}, ref_sd, spk_embed_integration_type="add")
    with pytest.raises(ic.InterchangeError):                                               # table size differs from n_speakers
        ic.from_espnet_state_dict({**esp, "sid_emb.weight": torch.zeros(9, 512)}, ref_sd, spk_embed_integration_type="add")
    with pytest.raises(ic.InterchangeError):                                               # a single-speaker model refuses a table
        base = TransformerTTS().state_dict()
        ic.from_espnet_state_dict({**ic.to_espnet_state_dict(base), "sid_emb.weight": torch.zeros(6, 512)}, base)
