"""Streaming inference against the whole-utterance call (B200, host clock + CUDA events).

    python scripts/bench_stream.py --out PATH   -> prints one line per case, writes PATH

Cases: B 1 / S 100 / T 800, B 64 / S 100 / T 800 and B 16 / S 300 / T 1600 (the planted stop head never fires, so every
utterance runs to T), each with chunk_frames 25, 50 and 100.  Per case, in one process:
  first_chunk_ms   host clock from the first next() of inference_stream() to the first chunk being ready (the driver
                   synchronises its side stream before yielding; the clock starts after a device synchronise)
  stream_ms        the whole stream drained, and inference_ms the whole-utterance inference(), device inputs; medians over
                   rounds that alternate the two after a warm-up
  emit_ms          CUDA-event time of each tts_decode_emit on the side stream (mean / max over one profiled stream)
  decode_step_us   decode kernel time per step from CUDA events around chunk_frames-step launches, in rotation: alone; with
                   the one emit of the previous chunk beside it, as inference_stream() runs them (the emit is much shorter than
                   the launch, so this average dilutes any contention over the whole launch); and with emits of that chunk
                   queued back to back on the side stream for the whole launch (every step shares L2 / HBM with an emit)
The card's name, power limit and maximum SM clock are read once with nvidia-smi --query-gpu in the same run.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import synthetic_state_dict  # noqa: E402
from transformer_tacotron2_b200 import TransformerTTS  # noqa: E402
from transformer_tacotron2_b200.model import postnet_halo  # noqa: E402

ROUNDS = int(os.environ.get("ROUNDS", "5"))
CASES = [(1, 100, 800), (64, 100, 800), (16, 300, 1600)]
CHUNKS = [25, 50, 100]


def inputs(B, S, seed):
    g = torch.Generator().manual_seed(seed)
    pl = ((torch.rand(B, generator=g) * 0.4 + 0.6) * S).floor().clamp(min=1).to(torch.int32); pl[0] = S
    ph = torch.randint(1, 128, (B, S), generator=g, dtype=torch.int64) * (torch.arange(S)[None, :] < pl[:, None])
    return ph.cuda(), pl.cuda()


def stream_once(m, ph, pl, T, chunk):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    it = m.inference_stream(ph, pl, max_len=T, seed=7, chunk_frames=chunk)
    next(it)
    t1 = time.perf_counter()
    for _ in it:
        pass
    torch.cuda.synchronize()
    return (t1 - t0) * 1e3, (time.perf_counter() - t0) * 1e3


def inference_once(m, ph, pl, T):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.inference(ph, pl, max_len=T, seed=7)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def decode_steps_with_and_without_emit(m, ph, pl, T, chunk, emit_ms):
    """Per-step decode kernel time of chunk-step launches, rotating: alone / one emit beside it / emits beside it throughout."""
    lib, h = m._lib, m._handle
    B, S = ph.shape
    halo = postnet_halo(m.cfg)
    ws = m._workspace(B, S, T)
    cur = torch.cuda.current_stream()
    side = torch.cuda.Stream()
    st, sd = C.c_void_p(cur.cuda_stream), C.c_void_p(side.cuda_stream)
    nbytes = lib.tts_stream_scratch_bytes(h, B, chunk + halo)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    ma = torch.empty(B, chunk + halo, 80, device="cuda"); sl = torch.empty(B, chunk + halo, device="cuda")
    assert lib.tts_decode_begin(h, ws.data_ptr(), B, S, T, 7, 0, st) == 0
    assert lib.tts_encode(h, ws.data_ptr(), ph.data_ptr(), pl.int().data_ptr(), B, S, T, None, st) == 0
    td, nf = C.c_int(0), C.c_int(0)
    assert lib.tts_decode_steps(h, ws.data_ptr(), chunk + halo, st) == 0
    times, k, emitted, launch_ms = ([], [], []), 0, 0, None
    while True:
        assert lib.tts_decode_status(h, ws.data_ptr(), C.byref(td), C.byref(nf), st) == 0
        if td.value + chunk > T:
            break
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        assert lib.tts_decode_steps(h, ws.data_ptr(), chunk, st) == 0
        e1.record(cur)
        frontier = td.value - halo
        mode = k % 3
        reps = 1 if mode == 1 else int(launch_ms / emit_ms) + 2 if mode == 2 else 0
        for _ in range(reps):
            assert lib.tts_decode_emit(h, ws.data_ptr(), scratch.data_ptr(), nbytes, max(emitted, frontier - chunk - halo), frontier,
                                       ma.data_ptr(), sl.data_ptr(), None, None, sd) == 0
        emitted = frontier
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if mode == 0:
            launch_ms = ms
        times[mode].append(ms * 1e3 / chunk)
        k += 1
    return tuple(statistics.median(t) for t in times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    m = TransformerTTS()
    m.load_state_dict(synthetic_state_dict().state_dict())
    results = []
    for B, S, T in CASES:
        ph, pl = inputs(B, S, 11)
        for chunk in CHUNKS:
            for _ in range(2):                                        # warm-up: module load, workspace, allocator
                stream_once(m, ph, pl, T, chunk)
                inference_once(m, ph, pl, T)
            first, total, whole = [], [], []
            for _ in range(ROUNDS):
                f, t = stream_once(m, ph, pl, T, chunk)
                first.append(f); total.append(t)
                whole.append(inference_once(m, ph, pl, T))
            m.profile_events = True
            m.emit_ms.clear()
            stream_once(m, ph, pl, T, chunk)
            m.profile_events = False
            emit = list(m.emit_ms)
            alone, beside, saturated = decode_steps_with_and_without_emit(m, ph, pl, T, chunk, statistics.mean(emit))
            r = dict(B=B, S=S, T=T, chunk_frames=chunk, first_chunk_ms=statistics.median(first),
                     stream_ms=statistics.median(total), inference_ms=statistics.median(whole),
                     stream_over_inference=statistics.median(total) / statistics.median(whole),
                     n_chunks=len(emit), emit_ms_mean=statistics.mean(emit), emit_ms_max=max(emit),
                     decode_step_us_alone=alone, decode_step_us_one_emit=beside, decode_step_us_emits_throughout=saturated)
            results.append(r)
            print(f"B {B:3d} S {S} T {T} chunk {chunk:3d}: first chunk {r['first_chunk_ms']:7.2f} ms | stream {r['stream_ms']:8.2f} ms vs "
                  f"inference {r['inference_ms']:8.2f} ms ({r['stream_over_inference']:.3f}x) | emit {r['emit_ms_mean']:.3f} ms mean "
                  f"({len(emit)} chunks) | decode step {alone:.1f} us alone, {beside:.1f} us with one emit, {saturated:.1f} us with emits "
                  f"throughout", flush=True)
    out = dict(gpu=gpu, rounds=ROUNDS, results=results)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=gpu)))


if __name__ == "__main__":
    main()
