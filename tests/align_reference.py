"""Reference for the cross-attention alignments and FastSpeech durations (test infrastructure).

cross_attention_weights() runs the oracle's teacher-forced forward and captures, with forward pre-hooks on every decoder
layer's cross-attention, the softmax probabilities that `MultiHeadAttention.attend` forms from the same inputs.  The hooks only
read their arguments, so the forward's outputs are unchanged.

durations_one() follows ESPnet's DurationCalculator (espnet2/tts/utils/duration_calculator.py) for one utterance: focus rate
F = mean over frames of max over phonemes, the (layer, head) with the largest F, durations = per-phoneme count of the frames
whose argmax is that phoneme.  durations_batch() applies it to every utterance of a batch, cut to its own lengths.
"""
import math

import torch


def cross_attention_weights(model, phonemes, phoneme_lens, mels, mel_lens, seed=0, utt_ids=None):
    """-> (P [L, B, H, T, S] fp32, zero at frames t >= mel_lens[b] and phonemes s >= phoneme_lens[b]; forward outputs)."""
    probs = []

    def hook(mod, args):
        xq, xkv, mask = args
        q, k = mod.split(mod.wq(xq)), mod.split(mod.wk(xkv))
        s = torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(mod.dh)
        probs.append(torch.softmax(s.masked_fill(~mask, float("-inf")), dim=-1).nan_to_num(0.0))

    handles = [layer.cross_attn.register_forward_pre_hook(hook) for layer in model.decoder.layers]
    try:
        with torch.no_grad():
            out = model(phonemes, phoneme_lens, mels, mel_lens, seed=seed, utt_ids=utt_ids)
    finally:
        for hd in handles:
            hd.remove()
    P = torch.stack(probs)
    T = P.shape[3]
    tvalid = torch.arange(T)[None, :] < mel_lens.to(torch.int64)[:, None]
    return P * tvalid[None, :, None, :, None], out


def durations_one(att_ws):
    """att_ws [L, H, T, S] of one utterance (its own lengths) -> (durations [S] int64, focus [L, H], chosen index l * H + h)."""
    L, H, T, S = att_ws.shape
    focus = att_ws.max(dim=-1)[0].mean(dim=-1)                        # [L, H]
    flat = att_ws.reshape(L * H, T, S)
    idx = int(focus.reshape(-1).argmax())                             # first maximum: lowest l * H + h on ties
    durations = torch.stack([flat[idx].argmax(-1).eq(i).sum() for i in range(S)]) if S else torch.zeros(0, dtype=torch.int64)
    return durations, focus, idx


def durations_batch(P, phoneme_lens, mel_lens, layers=None, fixed_head=None):
    """P [L, B, H, T, S] of the layers `layers` (default 0..L-1) -> (durations [B, S] int64, head [B] (= layer * H + h),
    focus [6, B, H] with -1 at unselected layers)."""
    L, B, H, T, S = P.shape
    layers = list(range(L)) if layers is None else list(layers)
    durs = torch.zeros(B, S, dtype=torch.int64)
    heads = torch.zeros(B, dtype=torch.int64)
    focus = torch.full((6, B, H), -1.0, dtype=torch.float64)
    for b in range(B):
        t, s = int(mel_lens[b]), int(phoneme_lens[b])
        d, f, idx = durations_one(P[:, b, :, :t, :s].double())
        focus[layers, b] = f
        if fixed_head is not None:
            li, h = layers.index(fixed_head // H), fixed_head % H
            idx = li * H + h
            d = torch.stack([P[li, b, h, :t, :s].argmax(-1).eq(i).sum() for i in range(s)])
        durs[b, :s] = d
        heads[b] = layers[idx // H] * H + idx % H
    return durs, heads, focus
