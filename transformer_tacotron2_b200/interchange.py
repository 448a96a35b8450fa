"""On-disk interchange (SURVEY.md 8(f)-4): import Transformer-TTS checkpoints written with ESPnet-style parameter names
(espnet2 `Transformer` TTS: `encoder.encoders.N.self_attn.linear_q`, `decoder.decoders.N.src_attn`, `feat_out`, `prob_out`,
`postnet.postnet.N.{0,1}`, scaled positional encodings `...embed.-1.alpha`) into this module's `state_dict` layout, and hand
mel-spectrograms to vocoders in the layout they expect.

Only POST-LayerNorm checkpoints can be imported (the oracle pins post-LN without final norms, SURVEY.md 8-P P1): a checkpoint that
carries `encoder.after_norm` / `decoder.after_norm` was trained with `normalize_before=True`, its arithmetic differs, and the import
refuses it instead of producing a model that silently computes something else.  The same holds for reduction factors != 1 and for
layer counts / widths other than the base model's.

Multi-speaker checkpoints (VCTK, LibriTTS, ...) carry a speaker-ID table `sid_emb.weight` and / or an x-vector projection
`projection.{weight,bias}`; they map to `speaker_embed.weight` / `spk_proj.*` of a model built with TTSConfig(n_speakers=...,
spk_embed_dim=...).  Only spk_embed_integration_type "add" is supported; language ids (`lid_emb`) and global style tokens (`gst`)
are refused."""
from __future__ import annotations

import re
from typing import Dict, Mapping, Optional

import torch


class InterchangeError(ValueError):
    pass


_ATT = {"linear_q": "wq", "linear_k": "wk", "linear_v": "wv", "linear_out": "wo"}
_FFN = {"w_1": "w1", "w_2": "w2"}


def _map_key(k: str) -> Optional[str]:
    """ESPnet-style key -> this module's key (None: the key carries no parameter we need, e.g. positional tables)."""
    m = re.fullmatch(r"encoder\.embed\.0\.embed\.weight", k)
    if m:
        return "enc_prenet.embed.weight"
    m = re.fullmatch(r"encoder\.embed\.0\.convs\.(\d+)\.(0|1)\.(weight|bias|running_mean|running_var|num_batches_tracked)", k)
    if m:
        i, which, p = m.groups()
        return f"enc_prenet.convs.{i}.{'conv' if which == '0' else 'bn'}.{p}"
    m = re.fullmatch(r"encoder\.embed\.0\.projection\.(weight|bias)", k)
    if m:
        return f"enc_prenet.proj.{m.group(1)}"
    if k == "encoder.embed.1.alpha":
        return "enc_alpha"
    if k == "decoder.embed.1.alpha":
        return "dec_alpha"
    m = re.fullmatch(r"encoder\.encoders\.(\d+)\.self_attn\.(linear_[qkv]|linear_out)\.(weight|bias)", k)
    if m:
        return f"encoder.layers.{m.group(1)}.self_attn.{_ATT[m.group(2)]}.{m.group(3)}"
    m = re.fullmatch(r"encoder\.encoders\.(\d+)\.feed_forward\.(w_[12])\.(weight|bias)", k)
    if m:
        return f"encoder.layers.{m.group(1)}.ffn.{_FFN[m.group(2)]}.{m.group(3)}"
    m = re.fullmatch(r"encoder\.encoders\.(\d+)\.norm([12])\.(weight|bias)", k)
    if m:
        return f"encoder.layers.{m.group(1)}.norm{m.group(2)}.{m.group(3)}"
    m = re.fullmatch(r"decoder\.embed\.0\.prenet\.(\d+)\.0\.(weight|bias)", k)
    if m:
        return f"dec_prenet.fc{int(m.group(1)) + 1}.{m.group(2)}"
    m = re.fullmatch(r"decoder\.embed\.0\.projection\.(weight|bias)", k)
    if m:
        return f"dec_prenet.proj.{m.group(1)}"
    m = re.fullmatch(r"decoder\.decoders\.(\d+)\.(self_attn|src_attn)\.(linear_[qkv]|linear_out)\.(weight|bias)", k)
    if m:
        att = "self_attn" if m.group(2) == "self_attn" else "cross_attn"
        return f"decoder.layers.{m.group(1)}.{att}.{_ATT[m.group(3)]}.{m.group(4)}"
    m = re.fullmatch(r"decoder\.decoders\.(\d+)\.feed_forward\.(w_[12])\.(weight|bias)", k)
    if m:
        return f"decoder.layers.{m.group(1)}.ffn.{_FFN[m.group(2)]}.{m.group(3)}"
    m = re.fullmatch(r"decoder\.decoders\.(\d+)\.norm([123])\.(weight|bias)", k)
    if m:
        return f"decoder.layers.{m.group(1)}.norm{m.group(2)}.{m.group(3)}"
    m = re.fullmatch(r"feat_out\.(weight|bias)", k)
    if m:
        return f"mel_linear.{m.group(1)}"
    m = re.fullmatch(r"prob_out\.(weight|bias)", k)
    if m:
        return f"stop_linear.{m.group(1)}"
    m = re.fullmatch(r"postnet\.postnet\.(\d+)\.(0|1)\.(weight|bias|running_mean|running_var|num_batches_tracked)", k)
    if m:
        i, which, p = m.groups()
        return f"postnet.convs.{i}.{'conv' if which == '0' else 'bn'}.{p}"
    if re.search(r"\.pe$", k) or k.endswith("num_batches_tracked"):
        return None
    return ""


_SPEAKER = {"sid_emb.weight": "speaker_embed.weight", "projection.weight": "spk_proj.weight", "projection.bias": "spk_proj.bias"}


def from_espnet_state_dict(src: Mapping[str, torch.Tensor], reference: Mapping[str, torch.Tensor],
                           spk_embed_integration_type: Optional[str] = None) -> Dict[str, torch.Tensor]:
    """Translate an ESPnet-style Transformer-TTS `state_dict` (optionally prefixed `tts.`) into this module's keys.
    `reference` = `TransformerTTS(cfg).state_dict()`: every target key must be produced with the reference's shape, and
    nothing the source contains may be left over.  Raises InterchangeError on anything that does not fit.

    A checkpoint with an x-vector projection (`projection.*`) needs spk_embed_integration_type="add", the value the ESPnet
    model was trained with: the weight shapes cannot tell "add" from "concat", and only "add" is this model's arithmetic."""
    if spk_embed_integration_type not in (None, "add"):
        raise InterchangeError(f"spk_embed_integration_type={spk_embed_integration_type!r} is not supported: only 'add' (the speaker "
                               "vector added to the encoder output) is this model's arithmetic")
    out: Dict[str, torch.Tensor] = {}
    unknown = []
    for k, v in src.items():
        k = k[4:] if k.startswith("tts.") else k
        if "after_norm" in k:
            raise InterchangeError("checkpoint was trained with normalize_before=True (pre-LayerNorm + final norm): only post-LayerNorm "
                                   "Transformer-TTS checkpoints are arithmetic-compatible with this model")
        if k.startswith("lid_emb."):
            raise InterchangeError("checkpoint has a language-ID embedding (lid_emb): multi-lingual models are not supported")
        if k.startswith("gst."):
            raise InterchangeError("checkpoint has global style tokens (gst): style-token conditioning is not supported")
        if k.startswith("projection.") and spk_embed_integration_type != "add":
            raise InterchangeError("checkpoint has an x-vector projection (projection.*): pass spk_embed_integration_type='add' if it was "
                                   "trained with the speaker vector added to the encoder output ('concat' is not supported)")
        t = _SPEAKER.get(k) or _map_key(k)
        if t is None:
            continue
        if t == "":
            unknown.append(k)
            continue
        v = v.detach().to(torch.float32)
        if t in ("enc_alpha", "dec_alpha"):
            v = v.reshape(())
        out[t] = v
    if unknown:
        raise InterchangeError(f"unrecognised parameters in the checkpoint: {unknown[:8]}{' ...' if len(unknown) > 8 else ''}")
    # ESPnet's convolutions before BatchNorm carry no bias; the BatchNorm bias absorbs it
    for k, r in reference.items():
        if k not in out and k.endswith(".conv.bias"):
            out[k] = torch.zeros_like(r, dtype=torch.float32)
        if k not in out and k.endswith("num_batches_tracked"):
            out[k] = r.clone()
    missing = [k for k in reference if k not in out]
    if missing:
        raise InterchangeError(f"checkpoint lacks parameters of the base model: {missing[:8]}{' ...' if len(missing) > 8 else ''}")
    for k, r in reference.items():
        if tuple(out[k].shape) != tuple(r.shape):
            raise InterchangeError(f"{k}: checkpoint shape {tuple(out[k].shape)} != base model {tuple(r.shape)} "
                                   "(reduction factor, width or layer count differs from the base Transformer-TTS)")
    extra = [k for k in out if k not in reference]
    if extra:
        raise InterchangeError(f"checkpoint has more layers than the base model: {extra[:8]}")
    return out


def to_espnet_state_dict(sd: Mapping[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """The inverse naming (for round trips and for handing trained weights to ESPnet-style tooling)."""
    inv: Dict[str, torch.Tensor] = {}
    att = {v: k for k, v in _ATT.items()}
    ffn = {v: k for k, v in _FFN.items()}
    for k, v in sd.items():
        if k == "enc_alpha":
            inv["encoder.embed.1.alpha"] = v.reshape(1); continue
        if k == "dec_alpha":
            inv["decoder.embed.1.alpha"] = v.reshape(1); continue
        k2 = k
        k2 = re.sub(r"^enc_prenet\.embed\.", "encoder.embed.0.embed.", k2)
        k2 = re.sub(r"^enc_prenet\.convs\.(\d+)\.conv\.", r"encoder.embed.0.convs.\1.0.", k2)
        k2 = re.sub(r"^enc_prenet\.convs\.(\d+)\.bn\.", r"encoder.embed.0.convs.\1.1.", k2)
        k2 = re.sub(r"^enc_prenet\.proj\.", "encoder.embed.0.projection.", k2)
        k2 = re.sub(r"^encoder\.layers\.(\d+)\.self_attn\.(w[qkvo])\.", lambda m: f"encoder.encoders.{m.group(1)}.self_attn.{att[m.group(2)]}.", k2)
        k2 = re.sub(r"^encoder\.layers\.(\d+)\.ffn\.(w[12])\.", lambda m: f"encoder.encoders.{m.group(1)}.feed_forward.{ffn[m.group(2)]}.", k2)
        k2 = re.sub(r"^encoder\.layers\.(\d+)\.norm", r"encoder.encoders.\1.norm", k2)
        k2 = re.sub(r"^dec_prenet\.fc(\d)\.", lambda m: f"decoder.embed.0.prenet.{int(m.group(1)) - 1}.0.", k2)
        k2 = re.sub(r"^dec_prenet\.proj\.", "decoder.embed.0.projection.", k2)
        k2 = re.sub(r"^decoder\.layers\.(\d+)\.(self_attn|cross_attn)\.(w[qkvo])\.",
                    lambda m: f"decoder.decoders.{m.group(1)}.{'self_attn' if m.group(2) == 'self_attn' else 'src_attn'}.{att[m.group(3)]}.", k2)
        k2 = re.sub(r"^decoder\.layers\.(\d+)\.ffn\.(w[12])\.", lambda m: f"decoder.decoders.{m.group(1)}.feed_forward.{ffn[m.group(2)]}.", k2)
        k2 = re.sub(r"^decoder\.layers\.(\d+)\.norm", r"decoder.decoders.\1.norm", k2)
        k2 = re.sub(r"^mel_linear\.", "feat_out.", k2)
        k2 = re.sub(r"^stop_linear\.", "prob_out.", k2)
        k2 = re.sub(r"^postnet\.convs\.(\d+)\.conv\.", r"postnet.postnet.\1.0.", k2)
        k2 = re.sub(r"^postnet\.convs\.(\d+)\.bn\.", r"postnet.postnet.\1.1.", k2)
        k2 = re.sub(r"^speaker_embed\.", "sid_emb.", k2)
        k2 = re.sub(r"^spk_proj\.", "projection.", k2)
        inv[k2] = v
    return inv


def mel_for_vocoder(mel: torch.Tensor, mel_lens: torch.Tensor, mean: Optional[torch.Tensor] = None, std: Optional[torch.Tensor] = None,
                    pad_value: float = 0.0) -> torch.Tensor:
    """[B, T, 80] (this module's output, zero past mel_lens) -> [B, 80, T] fp32, contiguous: the layout HiFi-GAN / WaveGlow /
    Parallel WaveGAN style vocoders take.  Optional de-normalisation with the training corpus' per-bin statistics (mel * std +
    mean); frames past each utterance's length are set to `pad_value` (the vocoder's silence level)."""
    x = mel.detach().to(torch.float32)
    if std is not None:
        x = x * std.to(x.device).view(1, 1, -1)
    if mean is not None:
        x = x + mean.to(x.device).view(1, 1, -1)
    T = x.shape[1]
    past = torch.arange(T, device=x.device)[None, :] >= mel_lens.to(x.device)[:, None]
    x = x.masked_fill(past[..., None], pad_value)
    return x.transpose(1, 2).contiguous()
