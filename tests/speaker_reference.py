"""Multi-speaker reference (test infrastructure): the oracle's TransformerTTS with ESPnet Transformer-TTS speaker conditioning,
spk_embed_integration_type "add" (espnet2/tts/transformer/transformer.py: `hs = hs + sid_emb(sids)`, then
`hs = hs + projection(F.normalize(spembs))`, before the decoder reads hs as memory):

    cond[b] = speaker_embed[sids[b]] + spk_proj(F.normalize(spembs[b]))      (each term present when configured)
    memory[b, s] = encoder_out[b, s] + cond[b]                                for EVERY s < S (padded keys are masked anyway)

It extends the oracle without changing it: the speaker modules are created after every base sub-module, so the base
parameters, their state_dict order and the canonical synthetic weights are those of the unconditioned oracle."""
from __future__ import annotations

from dataclasses import dataclass

import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import synthetic
from oracle.transformer_tts import TTSConfig, TransformerTTS


@dataclass(frozen=True)
class SpeakerTTSConfig(TTSConfig):
    n_speakers: int = 0
    spk_embed_dim: int = 0

    def base(self) -> TTSConfig:
        d = self.to_dict()
        d.pop("n_speakers"); d.pop("spk_embed_dim")
        return TTSConfig(**d)


class SpeakerTTS(TransformerTTS):
    """encode / forward / inference take sids [B] int and spembs [B, spk_embed_dim] float as keyword arguments."""

    def __init__(self, cfg: SpeakerTTSConfig):
        super().__init__(cfg)
        if cfg.n_speakers > 0:
            self.speaker_embed = nn.Embedding(cfg.n_speakers, cfg.d_model)
        if cfg.spk_embed_dim > 0:
            self.spk_proj = nn.Linear(cfg.spk_embed_dim, cfg.d_model)
        self._pending = None

    def speaker_cond(self, sids, spembs):
        """-> cond [B, 512] (None for an unconditioned model); ValueError on a missing or superfluous input."""
        c = self.cfg
        if (sids is not None) != (c.n_speakers > 0) or (spembs is not None) != (c.spk_embed_dim > 0):
            raise ValueError(f"sids / spembs do not fit n_speakers = {c.n_speakers}, spk_embed_dim = {c.spk_embed_dim}")
        cond = None
        if sids is not None:
            cond = self.speaker_embed(torch.as_tensor(sids).to(torch.int64))
        if spembs is not None:
            p = self.spk_proj(F.normalize(torch.as_tensor(spembs, dtype=torch.float32).detach()))
            cond = p if cond is None else cond + p
        return cond

    def encode(self, phonemes, phoneme_lens, seed: int = 0, utt_ids=None, sids=None, spembs=None):
        if self._pending is not None:                  # called from forward() / inference()
            sids, spembs = self._pending
        cond = self.speaker_cond(sids, spembs)
        hs = super().encode(phonemes, phoneme_lens, seed, utt_ids)
        return hs if cond is None else hs + cond[:, None, :]

    def _with_speakers(self, fn, sids, spembs, *a, **k):
        self.speaker_cond(sids, spembs)                # validate before any work
        self._pending = (sids, spembs)
        try:
            return fn(*a, **k)
        finally:
            self._pending = None

    def forward(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_ids=None, sids=None, spembs=None):
        return self._with_speakers(super().forward, sids, spembs, phonemes, phoneme_lens, mels, mel_lens, seed, utt_ids)

    def inference(self, phonemes, phoneme_lens, max_len: int = 800, seed: int = 0, utt_ids=None, return_before: bool = False,
                  sids=None, spembs=None):
        return self._with_speakers(super().inference, sids, spembs, phonemes, phoneme_lens, max_len, seed, utt_ids, return_before)


def make_speaker_model(cfg: SpeakerTTSConfig, stop_bias: float = -8.0, seed: int = synthetic.WEIGHT_SEED, zero: bool = False) -> SpeakerTTS:
    """The canonical synthetic model (oracle/synthetic.py: make_model, bit-identical base weights) plus speaker tables drawn with
    their default initialisation from seed + 2, rounded to bf16 like every other matrix (zero=True: all speaker tensors zero)."""
    base = synthetic.make_model(cfg.base(), stop_bias=stop_bias, seed=seed)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed + 2)
        m = SpeakerTTS(cfg)
    missing, unexpected = m.load_state_dict(base.state_dict(), strict=False)
    assert not unexpected and all(k.startswith(("speaker_embed.", "spk_proj.")) for k in missing), (missing, unexpected)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.startswith(("speaker_embed.", "spk_proj.")):
                p.copy_(torch.zeros_like(p) if zero else (p.to(torch.bfloat16).to(torch.float32) if p.dim() >= 2 else p))
    return m.eval()


def make_speakers(B: int, cfg: SpeakerTTSConfig, seed: int):
    """Mixed speakers for a batch: sids [B] int64 (None without a table), spembs [B, D] fp32 ~ N(0, 1) (None without a projection)."""
    g = torch.Generator().manual_seed(seed)
    sids = torch.randint(0, cfg.n_speakers, (B,), generator=g) if cfg.n_speakers > 0 else None
    spembs = torch.randn(B, cfg.spk_embed_dim, generator=g) if cfg.spk_embed_dim > 0 else None
    return sids, spembs
