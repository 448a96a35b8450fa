"""Streaming inference on the B200 (pytest -m gpu): TransformerTTS.inference_stream() and the tts_decode_emit entry point.

Concatenated chunks must equal inference() bit for bit.  That rests on gemm_tc_kernel reducing every output element in the same
tap / K order wherever its row sits in a tile and whichever N tile (128 or 256) launch_gemm_tc picks for the M at hand: a window
of a few dozen frames and the whole-utterance postnet generally take different tiles.  The first test pins that property."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


def _p(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def lib():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from transformer_tacotron2_b200 import _lib
    torch.zeros(1, device="cuda")
    return _lib.load()


def test_conv5_bits_independent_of_n_tile_and_row_position(lib):
    """conv k5 over 80 utterances x 128 frames takes the 256-wide N tile (m_tiles * 2 >= 148 SMs); the first 10 utterances alone
    take the 128-wide one; the same utterances cut to frames [40, 128) put every row at another position of its M tile."""
    g = torch.Generator().manual_seed(11)
    B, T, Cin, Cout = 80, 128, 512, 512
    X = (torch.randn(B, T, Cin, generator=g) * 0.5).to(torch.bfloat16).cuda()
    W = (torch.randn(5, Cout, Cin, generator=g) * 0.03).to(torch.bfloat16).cuda()
    bias = torch.randn(Cout, generator=g).cuda()

    def conv(x):
        b, t = x.shape[0], x.shape[1]
        x = x.contiguous()
        lens = torch.full((b,), t, dtype=torch.int32, device="cuda")
        y = torch.empty(b, t, Cout, device="cuda")
        assert lib.tts_k_conv5(_p(x), _p(W), _p(bias), _p(lens), _p(y), b, t, Cin, Cout, 2, _stream()) == 0
        torch.cuda.synchronize()
        return y

    full = conv(X)
    small = conv(X[:10])
    shifted = conv(X[:10, 40:])
    d_tile = float((full[:10] - small).abs().max())
    d_pos = float((shifted[:, 2:] - small[:, 42:]).abs().max())
    print(f"N tile 256 vs 128: max |diff| {d_tile:.3e}; row position shifted by 40: max |diff| {d_pos:.3e}")
    assert torch.equal(full[:10], small)
    assert torch.equal(shifted[:, 2:], small[:, 42:])


# ---------------------------------------------------------------------------------------------------------------------------
# end to end: inference_stream() against inference()
_MODELS = {}


def _model(stop_bias, G=0):
    from oracle import synthetic
    from tests.gpu_util import make_b200_model
    key = (stop_bias, G)
    if key not in _MODELS:
        _MODELS[key] = make_b200_model(synthetic.make_model(stop_bias=stop_bias), cluster_group=G)
    return _MODELS[key]


def _check_stream(g, ph, pl, max_len, seed, chunk, **kw):
    ref_a, ref_l, ref_s = g.inference(ph, pl, max_len=max_len, seed=seed, **kw)
    chunks = list(g.inference_stream(ph, pl, max_len=max_len, seed=seed, chunk_frames=chunk, **kw))
    B = ph.shape[0]
    pos = 0
    for ch in chunks:
        n = ch.mel_after.shape[1]
        assert ch.start == pos and n >= 1
        assert ch.mel_after.shape == (B, n, 80) and ch.stop_logits.shape == (B, n) and ch.n_valid.dtype == torch.int32
        assert ch.mel_after.device == ph.device and ch.finished.dtype == torch.bool
        pos += n
    assert chunks[-1].finished.all()
    ma = torch.cat([c.mel_after for c in chunks], 1)
    st = torch.cat([c.stop_logits for c in chunks], 1)
    nv = torch.stack([c.n_valid for c in chunks]).sum(0)
    assert ma.shape == ref_a.shape, (ma.shape, ref_a.shape)
    assert torch.equal(nv.to(ref_l.device, torch.int32), ref_l)
    assert torch.equal(st, ref_s)
    assert torch.equal(ma, ref_a), float((ma - ref_a).abs().max())
    for c in chunks:                                     # finished stays set once set; n_valid is the overlap with [0, len)
        want = (ref_l.to(c.n_valid.device) - c.start).clamp(0, c.mel_after.shape[1]).to(torch.int32)
        assert torch.equal(c.n_valid, want)
    return chunks


@pytest.mark.parametrize("B,S,max_len,chunk,stop_bias,G", [
    (1, 100, 800, 50, -8.0, 0),        # never stops: the session ends at max_len
    (64, 100, 800, 50, -8.0, 0),
    (13, 300, 200, 16, -0.45, 3),
    (5, 120, 300, 7, -0.45, 5),
    (5, 40, 60, 1, -0.45, 5),
    (13, 80, 120, 1000, -0.45, 3),     # chunk_frames > max_len: one chunk
    (1, 300, 800, 16, -0.45, 0),
    (64, 60, 160, 7, -0.45, 0),
])
def test_stream_equals_inference(lib, B, S, max_len, chunk, stop_bias, G):
    from oracle import synthetic
    ph, pl, _, _ = synthetic.make_inputs(B, S, 8, 900 + B + S, ragged=True)
    chunks = _check_stream(_model(stop_bias, G), ph.cuda(), pl.cuda(), max_len, 7, chunk)
    if chunk < max_len and chunks[-1].start > 0:
        assert chunks[0].mel_after.shape[1] == chunk


def test_stream_stop_cases(lib):
    """Utterances of one cluster group stop at different frames, some inside the halo of a chunk boundary."""
    import json
    import os
    from oracle import synthetic
    z = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "stop_cases.json")))
    for case in z["cases"]:
        ph, pl, _, _ = synthetic.make_inputs(z["B"], z["S"], 8, case["data_seed"], ragged=True)
        for G, chunk in ((5, 7), (3, 16), (5, 3)):
            g = _model(case["stop_bias"], G)
            _check_stream(g, ph.cuda(), pl.cuda(), z["max_len"], case["seed"], chunk)


def test_stream_budgets_and_utterance_ids(lib):
    from oracle import synthetic
    ph, pl, _, _ = synthetic.make_inputs(7, 24, 8, 503, ragged=True)
    budgets = torch.tensor([5, 24, 13, 1, 24, 17, 9], dtype=torch.int32)
    g = _model(-8.0)
    _check_stream(g, ph.cuda(), pl.cuda(), 24, 7, 4, max_lens=budgets)
    _check_stream(g, ph.cuda(), pl.cuda(), 24, 7, 3, utt_ids=[100, 7, 55, 3, 1000, 42, 8])
    _check_stream(_model(-0.45, 3), ph.cuda(), pl.cuda(), 40, 9, 5, utt_ids=[100, 7, 55, 3, 1000, 42, 8], max_lens=budgets + 10)


def test_stream_cpu_inputs_give_cpu_chunks(lib):
    from oracle import synthetic
    ph, pl, _, _ = synthetic.make_inputs(3, 30, 8, 77, ragged=True)
    _check_stream(_model(-0.45), ph, pl, 50, 3, 8)


# ---------------------------------------------------------------------------------------------------------------------------
# the C entry point
def _session(g, B, S, max_len, seed, data_seed):
    from oracle import synthetic
    lib, h = g._ensure_handle(), g._handle
    g.sync_weights()
    ph, pl, _, _ = synthetic.make_inputs(B, S, 8, data_seed, ragged=True)
    ph, pl = ph.cuda(), pl.cuda().int()
    ws = g._workspace(B, S, max_len)
    assert lib.tts_decode_begin(h, ws.data_ptr(), B, S, max_len, seed, 0, _stream()) == 0
    assert lib.tts_encode(h, ws.data_ptr(), ph.data_ptr(), pl.data_ptr(), B, S, max_len, None, _stream()) == 0
    return lib, h, ws, (ph, pl)


def _emit(lib, h, ws, B, t0, t1, scratch=None, nbytes=None):
    n = t1 - t0
    if scratch is None:
        nbytes = lib.tts_stream_scratch_bytes(h, B, n)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    ma = torch.empty(B, n, 80, device="cuda"); st = torch.empty(B, n, device="cuda"); mb = torch.empty(B, n, 80, device="cuda")
    ln = torch.empty(B, dtype=torch.int32, device="cuda")
    rc = lib.tts_decode_emit(h, ws.data_ptr(), scratch.data_ptr(), nbytes, t0, t1, ma.data_ptr(), st.data_ptr(), ln.data_ptr(),
                             mb.data_ptr(), _stream())
    torch.cuda.synchronize()
    return rc, ma, st, mb, ln


def test_emit_slices_equal_decode_end(lib):
    """After a completed decode, any [t_begin, t_end) equals that slice of tts_decode_end, launch count fixed per call."""
    B, S, max_len = 6, 40, 90
    g = _model(-0.45)
    lib, h, ws, keep = _session(g, B, S, max_len, 5, 61)
    td, nf = C.c_int(0), C.c_int(0)
    assert lib.tts_decode_steps(h, ws.data_ptr(), max_len, _stream()) == 0
    assert lib.tts_decode_status(h, ws.data_ptr(), C.byref(td), C.byref(nf), _stream()) == 0
    T = td.value
    ma = torch.empty(B, T, 80, device="cuda"); st = torch.empty(B, T, device="cuda"); mb = torch.empty(B, T, 80, device="cuda")
    ml = torch.empty(B, dtype=torch.int32, device="cuda")
    assert lib.tts_decode_end(h, ws.data_ptr(), T, ma.data_ptr(), ml.data_ptr(), st.data_ptr(), mb.data_ptr(), _stream()) == 0
    torch.cuda.synchronize()
    ranges = [(0, T), (0, 1), (T - 1, T), (3, 17), (11, 12), (9, T - 2), (T // 2, T)]
    for t0, t1 in [(t0, t1) for t0, t1 in ranges if 0 <= t0 < t1 <= T]:
        n0 = lib.tts_launch_count()
        rc, a, s, b, ln = _emit(lib, h, ws, B, t0, t1)
        assert rc == 0
        assert lib.tts_launch_count() - n0 == 6          # window kernel + five postnet GEMMs
        assert torch.equal(a, ma[:, t0:t1]) and torch.equal(s, st[:, t0:t1]) and torch.equal(b, mb[:, t0:t1]), (t0, t1)
        assert torch.equal(ln, ml)


def test_emit_validation(lib):
    from oracle import synthetic
    from tests.gpu_util import make_b200_model
    g = make_b200_model(synthetic.make_model(stop_bias=-8.0))
    B, S, max_len = 2, 20, 60
    g.sync_weights()
    lib, h = g._lib, g._handle
    ws = g._workspace(B, S, max_len)
    assert _emit(lib, h, ws, B, 0, 1)[0] == -2                 # no session
    lib, h, ws, keep = _session(g, B, S, max_len, 1, 5)
    assert _emit(lib, h, ws, B, 0, 1)[0] == -2                 # no status yet
    td, nf = C.c_int(0), C.c_int(0)
    assert lib.tts_decode_steps(h, ws.data_ptr(), 30, _stream()) == 0
    assert lib.tts_decode_status(h, ws.data_ptr(), C.byref(td), C.byref(nf), _stream()) == 0
    assert td.value == 30 and nf.value == 0
    assert lib.tts_decode_steps(h, ws.data_ptr(), 10, _stream()) == 0       # a later launch does not move the frontier
    assert _emit(lib, h, ws, B, 0, 21)[0] == -1                # past the frontier 30 - 10
    assert _emit(lib, h, ws, B, -1, 5)[0] == -1
    assert _emit(lib, h, ws, B, 7, 7)[0] == -1
    small = lib.tts_stream_scratch_bytes(h, B, 4)
    buf = torch.empty(small, dtype=torch.uint8, device="cuda")
    assert _emit(lib, h, ws, B, 0, 20, buf, small)[0] == -1    # scratch for 4 frames, window of 20 + halo
    assert _emit(lib, h, ws, B, 16, 20, buf, small)[0] == 0
    assert _emit(lib, h, ws, B, 0, 20)[0] == 0


def test_inference_launch_count_unchanged(lib):
    """inference(): encoder 48 + session init 1 + one decode launch + decode_end 7 (as before streaming existed)."""
    from oracle import synthetic
    g = _model(-8.0)
    ph, pl, _, _ = synthetic.make_inputs(3, 30, 8, 8, ragged=True)
    g.inference(ph.cuda(), pl.cuda(), max_len=20, seed=1)
    n0 = lib.tts_launch_count()
    g.inference(ph.cuda(), pl.cuda(), max_len=20, seed=1)
    assert lib.tts_launch_count() - n0 == 57


def test_early_close_leaves_the_module_usable(lib):
    from oracle import synthetic
    from tests.gpu_util import make_b200_model
    ph, pl, _, _ = synthetic.make_inputs(9, 50, 8, 31, ragged=True)
    ph, pl = ph.cuda(), pl.cuda()
    g = make_b200_model(synthetic.make_model(stop_bias=-0.45))
    fresh = make_b200_model(synthetic.make_model(stop_bias=-0.45))
    it = g.inference_stream(ph, pl, max_len=300, seed=4, chunk_frames=5)
    next(it); next(it)
    it.close()
    for x in g.inference_stream(ph, pl, max_len=300, seed=4, chunk_frames=5):
        break
    out = g.inference(ph, pl, max_len=300, seed=4)
    ref = fresh.inference(ph, pl, max_len=300, seed=4)
    for a, b in zip(out, ref):
        assert torch.equal(a, b)


def test_call_between_chunks_stops_the_stream(lib):
    """inference() between two chunks takes the workspace and the decode session: the open stream raises instead of yielding
    frames of the other call, and the call in between is unaffected."""
    from oracle import synthetic
    ph, pl, _, _ = synthetic.make_inputs(4, 40, 8, 33, ragged=True)
    ph, pl = ph.cuda(), pl.cuda()
    g = _model(-8.0)
    ref = g.inference(ph, pl, max_len=120, seed=2)
    it = g.inference_stream(ph, pl, max_len=120, seed=2, chunk_frames=10)
    first = next(it)
    assert torch.equal(first.mel_after, ref[0][:, :10])
    mid = g.inference(ph, pl, max_len=120, seed=2)
    for a, b in zip(mid, ref):
        assert torch.equal(a, b)
    with pytest.raises(RuntimeError, match="another call"):
        next(it)
