"""Cost of the cross-attention alignments and durations against the plain teacher-forced forward (B200, CUDA events).

    python scripts/bench_align.py [--out PATH]   -> prints one line per case, writes PATH (default align_bench.json)

Cases: B 64 / S 100 / T 800 and B 16 / S 300 / T 1600, ragged lengths.  Per case, in one process and alternating the modes
each round so that clock drift hits them alike:
  forward          TransformerTTS.forward (tts_forward: heads and postnet included)
  durations        TransformerTTS.durations: tts_forward_align without P and without heads / postnet
  P_1layer         TransformerTTS.alignments(layers=[2])
  P_6layers        TransformerTTS.alignments() (all six layers: 983 MB of fp32 at B 64 / T 800 / S 100)
and the alignment kernel alone (tts_k_cross_align on one layer's shapes, P written) with its write bandwidth, next to the
bandwidth of a device-to-device copy of the same byte count measured in the same run (read + write bytes over time).
P is larger than the 126 MB L2 at both shapes, so its stream goes to HBM.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import synthetic_state_dict  # noqa: E402
from transformer_tacotron2_b200 import TransformerTTS  # noqa: E402

ROUNDS = int(os.environ.get("ROUNDS", "10"))


def inputs(B, S, T, seed):
    g = torch.Generator().manual_seed(seed)
    pl = ((torch.rand(B, generator=g) * 0.4 + 0.6) * S).floor().clamp(min=1).to(torch.int32); pl[0] = S
    ml = ((torch.rand(B, generator=g) * 0.4 + 0.6) * T).floor().clamp(min=1).to(torch.int32); ml[0] = T
    ph = torch.randint(1, 128, (B, S), generator=g, dtype=torch.int64) * (torch.arange(S)[None, :] < pl[:, None])
    mels = torch.randn(B, T, 80, generator=g).clamp(-4, 4) * (torch.arange(T)[None, :] < ml[:, None])[..., None]
    return ph.cuda(), pl.cuda(), mels.cuda(), ml.cuda()


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def case(m, B, S, T):
    ph, pl, mels, ml = inputs(B, S, T, 11)
    modes = {
        "forward": lambda: m(ph, pl, mels, ml, seed=7),
        "durations": lambda: m.durations(ph, pl, mels, ml, seed=7),
        "P_1layer": lambda: m.alignments(ph, pl, mels, ml, seed=7, layers=[2]),
        "P_6layers": lambda: m.alignments(ph, pl, mels, ml, seed=7),
    }
    for f in modes.values():                                          # warm-up: module load, workspace, allocator
        f(); f()
    torch.cuda.synchronize()
    ms = {k: [] for k in modes}
    for _ in range(ROUNDS):
        for k, f in modes.items():
            ms[k].append(timed(f, 3))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}

    # the kernel alone, one layer, P written (random bf16 operands with the layer's shapes and the same ragged lengths)
    lib = m._lib
    Q = (torch.randn(B, T, 512, device="cuda") * 0.5).to(torch.bfloat16)
    K = (torch.randn(B, 8, S, 64, device="cuda") * 0.5).to(torch.bfloat16)
    P = torch.empty(B, 8, T, S, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    run = lambda: lib.tts_k_cross_align(Q.data_ptr(), 512, K.data_ptr(), ml.data_ptr(), pl.data_ptr(), B, 8, T, S,  # noqa: E731
                                        P.data_ptr(), None, None, st)
    assert run() == 0
    k_ms = sorted(timed(run, 20) for _ in range(5))[2]
    src, dst = torch.empty(P.numel(), device="cuda"), torch.empty(P.numel(), device="cuda")
    dst.copy_(src)
    c_ms = sorted(timed(lambda: dst.copy_(src), 20) for _ in range(5))[2]
    p_bytes = P.numel() * 4
    res = dict(B=B, S=S, T=T, rounds=ROUNDS, ms=med, ratio={k: med[k] / med["forward"] for k in med},
               P_bytes_per_layer=p_bytes, kernel_ms=k_ms, kernel_write_TBps=p_bytes / k_ms / 1e9,
               copy_ms=c_ms, copy_TBps_read_plus_write=2 * p_bytes / c_ms / 1e9)
    res["kernel_write_vs_copy"] = res["kernel_write_TBps"] / res["copy_TBps_read_plus_write"]
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="align_bench.json", help="where the JSON results go")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_align.py needs the GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("gpu:", smi)
    m = TransformerTTS()
    m.load_state_dict(synthetic_state_dict().state_dict())
    out = dict(gpu=smi, cases=[case(m, 64, 100, 800), case(m, 16, 300, 1600)])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
