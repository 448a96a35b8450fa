"""Cost of speaker conditioning: an unconditioned model against a multi-speaker one (n_speakers 256, x-vectors of 512, every
utterance of a batch with its own speaker) on the same base weights (B200, CUDA events).

    python scripts/bench_speakers.py [--out PATH]   -> prints one line per workload, writes PATH (default speakers_bench.json)

Workloads, ragged lengths, the two models alternated every round so that clock drift hits them alike:
  inference   B 64 / S 100 / 800 frames, TransformerTTS.inference (stop head planted never to fire: all 800 frames decode)
  forward     B 64 / S 100 / T 800, teacher-forced TransformerTTS.forward
  train_step  B 32 / S 100 / T 800, Trainer.step (forward, loss, backward, Adam; replayed from the captured CUDA graph)
Reported: median milliseconds per call of each model and the ratio conditioned / unconditioned, with the card's name and power
limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import synthetic_state_dict  # noqa: E402
from transformer_tacotron2_b200 import TTSConfig, TransformerTTS  # noqa: E402
from transformer_tacotron2_b200.training import Trainer  # noqa: E402

ROUNDS = int(os.environ.get("ROUNDS", "7"))
N_SPK, D_SPK = 256, 512


def inputs(B, S, T, seed):
    g = torch.Generator().manual_seed(seed)
    pl = ((torch.rand(B, generator=g) * 0.4 + 0.6) * S).floor().clamp(min=1).to(torch.int32); pl[0] = S
    ml = ((torch.rand(B, generator=g) * 0.4 + 0.6) * T).floor().clamp(min=1).to(torch.int32); ml[0] = T
    ph = torch.randint(1, 128, (B, S), generator=g, dtype=torch.int64) * (torch.arange(S)[None, :] < pl[:, None])
    mels = torch.randn(B, T, 80, generator=g).clamp(-4, 4) * (torch.arange(T)[None, :] < ml[:, None])[..., None]
    sids = torch.randint(0, N_SPK, (B,), generator=g, dtype=torch.int32)
    spembs = torch.randn(B, D_SPK, generator=g)
    return [t.cuda() for t in (ph, pl, mels, ml, sids, spembs)]


def models():
    base = synthetic_state_dict().state_dict()
    plain = TransformerTTS()
    plain.load_state_dict(base)
    torch.manual_seed(5)
    cond = TransformerTTS(TTSConfig(n_speakers=N_SPK, spk_embed_dim=D_SPK))
    sd = cond.state_dict()
    sd.update(base)
    cond.load_state_dict(sd)
    return plain, cond


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def run(name, calls):
    """calls: {"plain": fn, "cond": fn}; two warm-up calls each, then ROUNDS alternating timed calls."""
    for fn in calls.values():
        fn(); fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in calls}
    for _ in range(ROUNDS):
        for k, fn in calls.items():
            ms[k].append(timed(fn))
    med = {k: statistics.median(v) for k, v in ms.items()}
    res = dict(workload=name, plain_ms=med["plain"], cond_ms=med["cond"], ratio=med["cond"] / med["plain"],
               plain_all_ms=ms["plain"], cond_all_ms=ms["cond"])
    print(f"{name:11s} plain {med['plain']:9.3f} ms  conditioned {med['cond']:9.3f} ms  ratio {res['ratio']:.4f}", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="speakers_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_speakers.py measures the B200 path: no GPU")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    card = dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=smi.strip().splitlines()[0] if smi.strip() else "unavailable")
    print(card, flush=True)
    plain, cond = models()
    out = dict(card=card, rounds=ROUNDS, n_speakers=N_SPK, spk_embed_dim=D_SPK, results=[])
    with torch.no_grad():
        ph, pl, mels, ml, sids, sp = inputs(64, 100, 800, 1)
        out["results"].append(run("inference", {
            "plain": lambda: plain.inference(ph, pl, max_len=800, seed=7),
            "cond": lambda: cond.inference(ph, pl, max_len=800, seed=7, sids=sids, spembs=sp)}))
        out["results"].append(run("forward", {
            "plain": lambda: plain(ph, pl, mels, ml, seed=7),
            "cond": lambda: cond(ph, pl, mels, ml, seed=7, sids=sids, spembs=sp)}))
    ph, pl, mels, ml, sids, sp = inputs(32, 100, 800, 2)
    tp, tc = Trainer(plain), Trainer(cond)
    out["results"].append(run("train_step", {
        "plain": lambda: tp.step(ph, pl, mels, ml, seed=3),
        "cond": lambda: tc.step(ph, pl, mels, ml, seed=3, sids=sids, spembs=sp)}))
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
