#!/usr/bin/env python
"""bench.py -- batched autoregressive inference throughput (mel frames/s) of the B200 hot path.

Workload (BASELINE.json configs[2], the configuration the north-star target is quoted on): base
Transformer-TTS, batch 64 utterances x 100 phonemes -> 800 mel frames, greedy AR over the KV cache,
synthetic inputs, fixed random-init weights with a planted stop head that never fires (so every step
decodes all 800 frames).  A "step" is ONE whole inference of the batch: encoder + hoisted cross-K/V
projection + 800 decoder steps + postnet.  Multi-GPU: utterances are sharded across ranks with no
collective (weak scaling: 64 utterances per GPU; `--scaling strong` splits a fixed 64).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the oracle (CPU port; the reference ships no code) on host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed inference's outputs to DIR/*.npy (seeded inputs)

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (inputs already in HBM, CUDA-event
timed); `e2e` = the same through TransformerTTS.inference with HOST tensors (results land in the module's pinned
staging buffers, clone_outputs=False: the serving-loop form of the call; H2D + D2H inside the timed
region); `roofline` = the persistent decode kernel's algorithmic HBM bytes / its CUDA-event duration
against the measured copy bandwidth; `cpu_baseline` = the oracle on the box's host cores (bounded sample);
`train` = the other half of BASELINE.json's metric: utterances/s of the full train step (configs[3], B = 32 per GPU,
data parallel; the gradient exchange is fused into the optimiser kernel over NVLink peer memory), same timing rules.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W_BYTES = 44_663_970            # per-step decoder weight stream, bf16 (SURVEY.md 8(d))
STOP_BIAS = -8.0                # planted stop head: never fires
WEIGHT_SEED, DATA_SEED, DROPOUT_SEED = 1234, 103, 7


def decode_bytes(B: int, T: int, S: int) -> int:
    """Algorithmic HBM bytes of T decoder steps (SURVEY.md 8(d)): weights once per step, self-K/V rows
    0..t read + row t appended, cross-K/V read; bf16."""
    return T * W_BYTES + 12288 * B * (T * (T + 1) // 2 + T) + 12288 * B * S * T


def synthetic_state_dict():
    """Fixed random-init weights of the base architecture (no checkpoints exist): default nn inits under
    torch.manual_seed(1234), matrices rounded to bf16-representable values, stop bias planted."""
    from transformer_tacotron2_b200 import TransformerTTS
    rng = torch.get_rng_state()
    torch.manual_seed(WEIGHT_SEED)
    m = TransformerTTS()
    with torch.no_grad():
        for p in m.parameters():
            if p.dim() >= 2:
                p.copy_(p.to(torch.bfloat16).to(torch.float32))
        m.stop_linear.bias.fill_(STOP_BIAS)
        m.enc_alpha.fill_(0.5); m.dec_alpha.fill_(0.25)
    torch.set_rng_state(rng)
    return m


def synthetic_inputs(B: int, S: int, seed: int):
    g = torch.Generator().manual_seed(seed)
    ph = torch.randint(1, 128, (B, S), generator=g, dtype=torch.int64)
    return ph, torch.full((B,), S, dtype=torch.int32)


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir: str, utt0: int, mel_after, mel_lens, stop_logits):
    """Writes what one inference() call returned as float32 DIR/<name>.npy, so that two builds can be compared output for
    output.  Above DUMP_BYTES in all, a fixed seeded sample of utterances is written and their ids go to utterance_ids.npy."""
    import numpy as np
    B = mel_after.shape[0]
    per_utt = 4 * (mel_after[0].numel() + 1 + stop_logits[0].numel())
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES - 4096                                         # the .npy headers
    rows = torch.arange(B)
    if B * per_utt > budget:
        keep = budget // (per_utt + 8)                                 # 8 bytes per utterance id
        rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        np.save(os.path.join(out_dir, "utterance_ids.npy"), (rows + utt0).numpy().astype(np.float64))
    for name, t in (("mel_after", mel_after), ("mel_lens", mel_lens), ("stop_logits", stop_logits)):
        np.save(os.path.join(out_dir, name + ".npy"), t[rows.to(t.device)].float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        busy = [x for x in sm if smax and x > 0.3 * smax] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------
def cpu_oracle_sample(B: int, S: int, T: int, window: int, threads: int):
    """The oracle on host cores, bounded sample of the same workload: encoder once, `window` decoder
    steps at t ~ 0, T/2 and T-window (per-step cost is affine in t, so the three means integrate to
    the 800-step total), postnet once.  Returns (frames_per_s, description)."""
    from oracle import synthetic, TransformerTTS as Oracle
    torch.set_num_threads(threads)
    o = Oracle().eval()
    o.load_state_dict(synthetic_state_dict().state_dict())
    ph, pl = synthetic_inputs(B, S, DATA_SEED)
    import numpy as np
    b_ids = np.arange(B)
    with torch.no_grad():
        t0 = time.perf_counter(); mem = o.encode(ph, pl); t_enc = time.perf_counter() - t0
        state = o.init_decode_state(mem, pl, T)
        g = torch.Generator().manual_seed(1)
        for l in range(len(state["sk"])):                       # contents do not matter for timing
            state["sk"][l].copy_(torch.randn(state["sk"][l].shape, generator=g) * 0.5)
            state["sv"][l].copy_(torch.randn(state["sv"][l].shape, generator=g) * 0.5)
        means, starts = [], [0, max(0, T // 2 - window // 2), max(0, T - window)]
        frame = torch.zeros(B, 1, 80)
        o.decode_step(state, frame, 0, DROPOUT_SEED, b_ids)      # warm-up
        for st in starts:
            t0 = time.perf_counter()
            for t in range(st, min(T, st + window)):
                frame, _ = o.decode_step(state, frame, t, DROPOUT_SEED, b_ids)
            means.append((time.perf_counter() - t0) / max(1, min(T, st + window) - st))
        mids = [s + window / 2 for s in starts]
        # least-squares line through the three (t, sec/step) points, summed over t = 0..T-1
        n = len(mids); mx = sum(mids) / n; my = sum(means) / n
        slope = sum((x - mx) * (y - my) for x, y in zip(mids, means)) / max(1e-12, sum((x - mx) ** 2 for x in mids))
        icpt = my - slope * mx
        t_dec = sum(icpt + slope * t for t in range(T))
        mel = torch.randn(B, T, 80, generator=g)
        lens = torch.full((B,), T, dtype=torch.int32)
        t0 = time.perf_counter(); o._postnet(mel, lens, DROPOUT_SEED, b_ids); t_post = time.perf_counter() - t0
    total = t_enc + t_dec + t_post
    desc = (f"oracle fp32, {threads} threads: encoder + {window}-step windows at t={starts} (affine fit, summed over {T} steps) "
            f"+ postnet; est. {total:.1f} s per {B}x{T} batch (enc {t_enc:.2f}, dec {t_dec:.1f}, post {t_post:.2f})")
    return B * T / total, desc


def run_reference(args, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    B, S, T = args.batch, args.phonemes, args.frames
    vals = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        v, desc = cpu_oracle_sample(B, S, T, window=args.ref_window, threads=threads)
        if i >= args.warmup:
            vals.append((v, time.perf_counter() - t0))
    value = statistics.mean(v for v, _ in vals)
    line = {
        "impl": "reference", "metric": "mel frames/s, batched AR inference", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * B * T / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"configs[2]: base model batched greedy AR inference, B={B}, S={S}, {T} frames (CPU oracle; reference ships no code)",
                   "batch_per_gpu": B, "phonemes": S, "frames": T},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist
    from transformer_tacotron2_b200 import _lib
    import datetime
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from transformer_tacotron2_b200 import _lib as _libmod
    if world > 1:
        # NCCL announces its version on stdout when the first communicator is created; stdout carries the ONE JSON line of this
        # run, so file descriptor 1 points at stderr until the communicator exists
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            # short collective timeout: a rank that dies must not park its peers in a barrier for the default 10 minutes
            dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=args.nccl_timeout))
            if local_rank == 0:                                     # one builder per node, then everybody loads the finished library
                _libmod.load()
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    T, S = args.frames, args.phonemes
    B = args.batch if args.scaling == "weak" else max(1, args.batch // world)
    utt0 = rank * B
    src = synthetic_state_dict()
    from transformer_tacotron2_b200 import TransformerTTS
    model = TransformerTTS(device=local_rank)
    model.load_state_dict(src.state_dict())
    model.sync_weights()
    lib = _lib.load()
    extra = {}
    ph_all, pl_all = synthetic_inputs(B * world, S, DATA_SEED)
    ph, pl = ph_all[utt0:utt0 + B].contiguous(), pl_all[utt0:utt0 + B].contiguous()
    ph_d, pl_d = ph.to(dev), pl.to(dev)
    ph_pin, pl_pin = ph.pin_memory(), pl.pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    model.profile_events = True
    # ---- device-resident: inputs already in HBM ------------------------------------------------
    for _ in range(args.warmup):
        out = model.inference(ph_d, pl_d, max_len=T, seed=DROPOUT_SEED, utt_offset=utt0)
    assert out[0].shape == (B, T, 80) and int(out[1].min()) == T, "planted stop head fired: not the named workload"
    model.decode_ms.clear()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = lib.tts_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = model.inference(ph_d, pl_d, max_len=T, seed=DROPOUT_SEED, utt_offset=utt0)
    e1.record()
    barrier()
    launches = lib.tts_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    dec_ms = max_over_ranks(statistics.mean(model.decode_ms))
    frames_total = world * B * T * args.steps
    value = frames_total / (dev_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, utt0, *out)

    # ---- end to end through the public API with HOST tensors -----------------------------------
    model.profile_events = False
    for _ in range(max(1, args.warmup // 2)):
        model.inference(ph_pin, pl_pin, max_len=T, seed=DROPOUT_SEED, utt_offset=utt0, clone_outputs=False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ma, ml, st = model.inference(ph_pin, pl_pin, max_len=T, seed=DROPOUT_SEED, utt_offset=utt0, clone_outputs=False)
    torch.cuda.synchronize(dev)
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e = frames_total / e2e_s
    h2d = B * S * 8 + B * 4
    d2h = B * T * 80 * 4 + B * T * 4 + B * 4

    # ---- the other configurations of BASELINE.json, same timing rules, each with its own decode-kernel roofline ---------------
    def measure_case(name, Bc, Sc, Tc, utt_off, steps, desc):
        """device-resident inference of Bc utterances on THIS rank -> (ms per inference, decode-kernel ms)"""
        phc, plc = synthetic_inputs(Bc, Sc, DATA_SEED + 17)
        phc, plc = phc.to(dev), plc.to(dev)
        model.profile_events = True
        for _ in range(3):
            o = model.inference(phc, plc, max_len=Tc, seed=DROPOUT_SEED, utt_offset=utt_off)
        assert int(o[1].min()) == Tc
        model.decode_ms.clear()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            model.inference(phc, plc, max_len=Tc, seed=DROPOUT_SEED, utt_offset=utt_off)
        b.record()
        barrier()
        ms = max_over_ranks(a.elapsed_time(b)) / steps
        dms = max_over_ranks(statistics.mean(model.decode_ms))
        model.profile_events = False
        return ms, dms

    def case_line(desc, Bc, Sc, Tc, nranks, ms, dms):
        peak_, _k = measured_peaks()
        algo_ = decode_bytes(Bc, Tc, Sc)
        ach = algo_ / (dms * 1e-3) / 1e9
        return {"value": nranks * Bc * Tc / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "config": {"workload": desc, "batch_per_gpu": Bc, "phonemes": Sc, "frames": Tc},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak_, "unit": "GB/s", "frac": ach / peak_, "algorithmic_bytes_per_launch": algo_,
                             "kernel_ms_per_launch": dms, "us_per_decoder_step": 1e3 * dms / Tc}}

    if not args.no_extra:
        ksteps = max(2, args.steps // 4)
        # configs[2] as BASELINE.json words it: a FIXED batch of 64 utterances sharded over the N GPUs (strong scaling)
        Bs = max(1, args.batch // world)
        ms, dms = measure_case("strong", Bs, S, T, rank * Bs, ksteps, "")
        extra["strong"] = case_line(f"configs[2] strong scaling: 64 utterances sharded over {world} GPU(s), {Bs} per GPU, S={S}, {T} frames", Bs, S, T, world, ms, dms)
        extra["strong"]["scaling"] = "strong"
        # configs[1]: batch-1 latency path (every rank decodes one utterance; value = one GPU's frames/s, latency per frame beside it)
        ms, dms = measure_case("latency_b1", 1, S, T, rank, ksteps, "")
        extra["latency_b1"] = case_line(f"configs[1]: greedy AR, batch 1, S={S}, {T} frames, latency path (per GPU)", 1, S, T, 1, ms, dms)
        extra["latency_b1"]["us_per_frame"] = 1e3 * ms / T
        # configs[4]: long utterances, batch 16 per GPU, 300 phonemes -> 1600 frames
        ms, dms = measure_case("long", 16, 300, 1600, rank * 16, 2, "")
        extra["long"] = case_line("configs[4]: long-utterance inference, B=16/GPU, S=300, 1600 frames", 16, 300, 1600, world, ms, dms)

    if not args.no_extra:
        # SURVEY.md 8(f)-2/3: a ragged batch (256 utterances per GPU, frame budgets U[0.6, 1] x T) -- valid frames / s with the
        # batch decoded in the caller's order on statically assigned clusters, and sorted by length with clusters stealing groups
        Br = 256
        phr, plr = synthetic_inputs(Br, S, DATA_SEED + 29)
        phr, plr = phr.to(dev), plr.to(dev)
        gen = torch.Generator().manual_seed(DATA_SEED + 31 + rank)
        budgets = (T * (0.6 + 0.4 * torch.rand(Br, generator=gen))).to(torch.int32).clamp(1, T).to(dev)
        valid = int(budgets.sum())
        res = {}
        for name, kw in (("unsorted_static", dict(sort_by_length=False, work_stealing=False)), ("sorted_stealing", dict(sort_by_length=True, work_stealing=True))):
            for _ in range(2):
                o = model.inference(phr, plr, max_len=T, seed=DROPOUT_SEED, utt_offset=rank * Br, max_lens=budgets, **kw)
            assert o[1].tolist() == budgets.tolist()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(2):
                model.inference(phr, plr, max_len=T, seed=DROPOUT_SEED, utt_offset=rank * Br, max_lens=budgets, **kw)
            b.record()
            barrier()
            res[name] = world * valid / (max_over_ranks(a.elapsed_time(b)) / 2 * 1e-3)
        extra["ragged"] = {"value": res["sorted_stealing"], "unit": "valid frames/s", "unsorted_static": res["unsorted_static"],
                           "config": {"workload": f"ragged batch: {Br} utterances/GPU, S={S}, frame budgets U[0.6,1] x {T} (mean {valid / Br:.0f}), "
                                                  "length-sorted groups + device-side group queue vs caller order + static clusters"}}

    # ---- second half of BASELINE.json's metric: teacher-forced train step (configs[3]: B = 32 per GPU, data parallel,
    #      one NCCL all-reduce over the flat gradient buffer per step), utterances / s over all ranks -------------------
    train = None
    if not args.no_train:
        from transformer_tacotron2_b200.training import Trainer
        Bt, Tt = args.train_batch, T
        tr = Trainer(model, lr=1e-4, world_size=world, rank=rank)
        g = torch.Generator().manual_seed(DATA_SEED + 1000 + rank)
        tph = torch.randint(1, 128, (Bt, S), generator=g).to(dev); tpl = torch.full((Bt,), S, dtype=torch.int32, device=dev)
        tmel = torch.randn(Bt, Tt, 80, generator=g).clamp(-4, 4).to(dev); tml = torch.full((Bt,), Tt, dtype=torch.int32, device=dev)
        for i in range(args.warmup):
            tr.step(tph, tpl, tmel, tml, seed=DROPOUT_SEED + i, utt_offset=rank * Bt)
        barrier()
        launches_t0 = lib.tts_launch_count()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for i in range(args.steps):
            loss = tr.step(tph, tpl, tmel, tml, seed=DROPOUT_SEED + 100 + i, utt_offset=rank * Bt)
        t1e.record()
        barrier()
        train_ms = max_over_ranks(t0e.elapsed_time(t1e)) / args.steps
        # tensor roofline of the step: algorithmic FLOPs = 3 x forward (SURVEY.md 8(d): 28.14 / 52.88 GF per utterance at
        # S = 100, T = 400 / 800; backward = 2 x forward) against the measured sustained bf16 rate
        fwd_gf = {400: 28.14, 800: 52.88}.get(Tt) if S == 100 else None
        tpeak = None
        try:
            tpeak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
        except Exception:
            tpeak = None
        troof = None
        if fwd_gf and tpeak:
            ach = 3.0 * fwd_gf * Bt / (train_ms * 1e-3) / 1e3
            troof = {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak,
                     "algorithmic_gflop_per_step_per_gpu": 3.0 * fwd_gf * Bt}
        train = {"metric": "utterances/s, teacher-forced train step (forward + loss + backward + all-reduce + Adam)",
                 "value": world * Bt / (train_ms * 1e-3), "unit": "utt/s", "ms_per_step": train_ms, "loss": float(loss),
                 "gpu_launches_per_step": int((lib.tts_launch_count() - launches_t0) // args.steps), "roofline": troof,
                 "l2": "per-step working set (4.3 GB of saved activations + 0.85 GB of optimiser state) exceeds the 126 MB L2; no flush needed",
                 "config": {"workload": f"configs[3]: base model train step, B={Bt}/GPU, S={S}, T={Tt}, bf16 operands / fp32 accumulate, "
                                        f"fp32 master + Adam, data parallel x{world} "
                                        + ("(gradient exchange fused into the optimiser kernel: reduce-scatter by NVLink peer loads -> Adam on the "
                                           "rank's shard -> all-gather by peer stores)" if tr._peers else "(single rank: no exchange)" if world == 1
                                           else "(one NCCL all-reduce over 53.0 M fp32 gradients)")}}
        tr = None

    if rank != 0:
        return
    peak, peak_kind = measured_peaks()
    algo = decode_bytes(B, T, S)
    achieved = algo / (dec_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "decode_kernel_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    line = {
        "metric": "mel frames/s, batched AR inference", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"configs[2]: base model batched greedy AR inference, B={B}/GPU, S={S}, {T} frames, KV cache; "
                               "one step = encoder + cross-KV + decode loop + postnet",
                   "batch_per_gpu": B, "phonemes": S, "frames": T, "parallelism": f"utterance-sharded x{world}, no collective",
                   "l2": "per-step KV working set (up to 708 MB) exceeds the 126 MB L2; no flush needed",
                   "weights": "random-init (seed 1234), stop head planted so no utterance stops early"},
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "decode_cluster_kernel (persistent 8-CTA clusters, all decoder steps of one batch in one launch)",
                     "achieved": achieved, "peak": peak, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})", "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes_per_launch": algo,
                     "kernel_ms_per_launch": dec_ms, "us_per_decoder_step": 1e3 * dec_ms / T},
        "clocks": clocks,
    }
    if train is not None:
        line["train"] = train
    line.update(extra)
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, desc = cpu_oracle_sample(B, S, T, window=args.cpu_window, threads=threads)
        line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": threads, "kind": "port", "sample": desc}
        if not args.no_cpu_full_b1:
            # how good is the sampled estimate?  configs[1] (batch 1, 800 frames) is short enough to run IN FULL on the CPU:
            # time it, and put the affine 3-window estimate of the same workload beside it
            from oracle import TransformerTTS as Oracle
            torch.set_num_threads(threads)
            o = Oracle().eval(); o.load_state_dict(synthetic_state_dict().state_dict())
            ph1, pl1 = synthetic_inputs(1, S, DATA_SEED)
            t0 = time.perf_counter()
            with torch.no_grad():
                o1 = o.inference(ph1, pl1, max_len=T, seed=DROPOUT_SEED)
            full_s = time.perf_counter() - t0
            est_v, _ = cpu_oracle_sample(1, S, T, window=args.cpu_window, threads=threads)
            line["cpu_baseline"]["full_run_b1"] = {"frames_per_s": T / full_s, "seconds": full_s, "frames": int(o1[1][0]),
                                                   "sampled_estimate_frames_per_s": est_v, "estimate_over_full": est_v / (T / full_s),
                                                   "note": "configs[1] run in full on the host cores (oracle, fp32) next to the 3-window affine estimate of the same workload"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", type=int, default=800)
    ap.add_argument("--phonemes", type=int, default=100)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-window", type=int, default=50)
    ap.add_argument("--ref-window", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-full-b1", action="store_true", help="skip the full CPU run of configs[1] that validates the sampled estimate")
    ap.add_argument("--no-train", action="store_true", help="skip the train-step measurement (the `train` key)")
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--no-extra", action="store_true", help="skip the strong-scaling / batch-1 latency / long-utterance lines")
    ap.add_argument("--nccl-timeout", type=int, default=180, help="seconds before a collective gives up (a dead rank must not stall the job)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed inference returned on "
                    "rank 0 (mel_after, mel_lens, stop_logits) to DIR/<name>.npy as float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3                                             # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args, rank)
        return
    try:
        run_b200(args, rank, world, local_rank)
    except BaseException:
        import traceback
        traceback.print_exc()
        sys.stderr.flush(); sys.stdout.flush()
        os._exit(1)                                                 # fail fast: no barrier, no destroy_process_group on a broken context
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
