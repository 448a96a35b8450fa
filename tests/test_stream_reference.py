"""CPU: the arithmetic streaming inference rests on.  The eval-mode postnet run window by window, each window carrying `halo`
frames of context on both sides, gives the whole-utterance postnet's output on the window's centre; and the decode / emit
schedule of TransformerTTS.inference_stream() tiles the output exactly without emitting a frame whose postnet context is not
decoded yet."""
import numpy as np
import pytest
import torch

from transformer_tacotron2_b200.model import StreamSchedule, TTSConfig, postnet_halo

HALO = postnet_halo(TTSConfig())


def test_halo_is_ten_frames():
    assert HALO == 10


@pytest.fixture(scope="module")
def oracle():
    from oracle import synthetic
    return synthetic.make_model(stop_bias=-8.0).eval()


def _window(o, mel, lens, t_status, t_begin, t_end):
    """What tts_decode_emit computes for frames [t_begin, t_end) when t_status frames are decoded: the postnet over frames
    [a, e) only, zero outside them, each utterance masked at min(lens, t_status) - a."""
    a, e = max(0, t_begin - HALO), min(t_end + HALO, t_status)
    L = (torch.minimum(lens, torch.tensor(t_status)) - a).clamp(0, e - a)
    m = (torch.arange(e - a)[None, :] < L[:, None]).float()[..., None]
    x = mel[:, a:e] * m
    out = (x + o._postnet(x, L, 0, np.arange(mel.shape[0]))) * m
    return out[:, t_begin - a:t_end - a]


def _full(o, mel, lens):
    T = mel.shape[1]
    m = (torch.arange(T)[None, :] < lens[:, None]).float()[..., None]
    x = mel * m
    return (x + o._postnet(x, lens, 0, np.arange(mel.shape[0]))) * m


@torch.no_grad()
def test_windowed_postnet_equals_full(oracle):
    g = torch.Generator().manual_seed(3)
    B, T = 4, 67
    mel = torch.randn(B, T, 80, generator=g)
    lens = torch.tensor([67, 40, 1, 55])
    ref = _full(oracle, mel, lens)
    ranges = [(0, 1), (0, 67), (66, 67), (0, 13), (13, 14), (5, 30), (30, 61), (39, 41), (54, 56), (50, 67), (20, 21)]
    for t0, t1 in ranges:
        got = _window(oracle, mel, lens, T, t0, t1)
        assert torch.allclose(got, ref[:, t0:t1], rtol=1e-5, atol=1e-5), (t0, t1, float((got - ref[:, t0:t1]).abs().max()))
        assert not got[2, max(0, 1 - t0):].any() and not got[1, max(0, 40 - t0):].any()        # zero past each utterance's end


@torch.no_grad()
def test_window_longer_than_the_utterance(oracle):
    """T = 7 < 2 * halo + 1: every window reaches both true edges."""
    g = torch.Generator().manual_seed(4)
    mel = torch.randn(2, 7, 80, generator=g)
    lens = torch.tensor([7, 3])
    ref = _full(oracle, mel, lens)
    for t0, t1 in ((0, 7), (3, 4), (0, 1), (6, 7)):
        assert torch.allclose(_window(oracle, mel, lens, 7, t0, t1), ref[:, t0:t1], rtol=1e-5, atol=1e-5)


@torch.no_grad()
def test_frames_past_the_decode_point_do_not_reach_the_frontier(oracle):
    """Mid-decode (t_status frames decoded, frames past it still garbage), frames below t_status - halo are already final."""
    g = torch.Generator().manual_seed(5)
    B, T, t_status = 3, 90, 61
    mel = torch.randn(B, T, 80, generator=g)
    lens = torch.tensor([90, 30, 75])                    # utterance 1 has stopped; 0 and 2 run past t_status
    ref = _full(oracle, mel, lens)
    seen = mel.clone()
    seen[:, t_status:] = 1e3 * torch.randn(B, T - t_status, 80, generator=g)
    for t0, t1 in ((0, t_status - HALO), (40, t_status - HALO), (t_status - HALO - 1, t_status - HALO)):
        assert torch.allclose(_window(oracle, seen, lens, t_status, t0, t1), ref[:, t0:t1], rtol=1e-5, atol=1e-5)


def _simulate(lens, max_len, chunk):
    """Drive StreamSchedule with a model of the decode loop: each launch runs `steps` more frames (up to max_len); tts_decode_status
    reports the longest utterance once every one has stopped.  lens[b] = frame count of utterance b (max_len: never stops)."""
    sched = StreamSchedule(chunk, HALO, max_len)
    t, B = 0, len(lens)
    pending = sched.first_steps()
    chunks = []
    while True:
        t = min(t + pending, max_len)
        nf = sum(1 for v in lens if v <= t)
        ended = nf >= B or t >= max_len
        t_done = max(lens) if nf >= B else t
        pending, rng = sched.after_status(t_done, ended)
        if rng is not None:
            t0, t1 = rng
            assert t1 - t0 <= sched.max_emit_frames()
            for v in lens:                               # a running utterance: nothing within halo of the decode point
                if v > t_done:
                    assert t1 <= t_done - HALO
            chunks.append(rng)
        if ended:
            return chunks, t_done


@pytest.mark.parametrize("chunk", [1, 7, 16, 50, 1000])
@pytest.mark.parametrize("lens,max_len", [([800], 800), ([3], 800), ([11], 40), ([12, 57, 3, 800], 800), ([1], 1), ([9, 25], 30),
                                          ([60, 61, 62], 200), ([21, 20], 100)])
def test_schedule_tiles_the_output(lens, max_len, chunk):
    chunks, t_out = _simulate(lens, max_len, chunk)
    assert t_out == max(lens)
    assert chunks[0][0] == 0 and chunks[-1][1] == max(lens)
    for (a0, a1), (b0, b1) in zip(chunks, chunks[1:]):
        assert a1 == b0 and a0 < a1
    if chunk < max_len and max(lens) > chunk + 2 * HALO:
        assert chunks[0] == (0, chunk)                   # first chunk: chunk + halo decoder steps


def test_schedule_rejects_empty_chunks():
    with pytest.raises(ValueError):
        StreamSchedule(0, HALO, 10)
