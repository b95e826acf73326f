"""One wideband input's channels demodulated on several GPUs (ba_cuda_create_multi_split) against a plain engine, on cfg4.

Input: configs.cfg4 (one 61.44 Msps cf32 stream, fft 8192, 2000 mixed AM/NFM channels), device-resident: a seeded 2 s
template synthesised on each GPU that homes the input, repeated to cover the run.  Audio goes to the engine's pinned host
memory.  One step is one second of signal (8 batches); three tickets are kept in flight as in bench.py.  Timing is wall
time around the timed steps, which end in a wait for the last ticket, plus CUDA events inside the engine (kernel_ms).

Arms, each `--steps` timed steps after `--warmup` steps:
  (a) a plain engine on GPU 0
  (b) create_multi_split over [0] (every channel at home: the group only forwards calls), alternated with (a) `--reps` times
  (c) create_multi_split over [0, 0], channels alternately on the two members: the ship/gather overhead on shared SMs
  (d) with G >= 2 visible GPUs: over all of them, channel c on GPU c % G
Per arm: ms per step, x real time, the channelizer's and the demodulator's event times per step (the maximum over members:
the C-ABI reports a group's timings as the maximum), the ship and gather bytes per step computed from the shapes, and a
digest of every output of the warm-up steps (audio and status), which must be equal across arms.

Prints one JSON line and writes it to profiles/r04_bench_split_device.json (or --out).
Usage: python tools/bench_split_device.py [--steps 20] [--warmup 3] [--reps 3] [--out PATH]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

DEPTH = 3
TEMPLATE_S = 2.0


def gpu_facts():
    import torch
    facts = {"gpu": torch.cuda.get_device_name(0), "visible_gpus": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        facts["power_limit_and_max_sm_clock"] = [ln.strip() for ln in q.stdout.strip().splitlines()]
    except (OSError, subprocess.SubprocessError) as ex:
        facts["power_limit_and_max_sm_clock"] = "not read: %s" % ex
    return facts


def traffic(cfg, gpu_of_channel, home=0):
    """Bytes per one-second step between GPUs, from the shapes: to the followers the magnitudes (4 B per frame) of every
    channel away from home plus the picked IQ (8 B per frame) of those that read raw IQ (NFM, low-pass); back to the home
    the audio (4 B per sample), the status (40 B per batch) and iq_out (8 B per sample) of those channels."""
    from boondock_airband_b200 import abi
    dev = cfg.devices[0]
    frames = cfg.wave_rate  # frames per second of signal
    ship = gather = 0
    for c, ch in enumerate(dev.channels):
        if gpu_of_channel is None or gpu_of_channel[c] == home:
            continue
        raw = ch.modulation == "nfm" or ch.bandwidth != 0 or ch.has_iq_outputs or (cfg.flags & abi.FLAG_KEEP_PICKS)
        ship += frames * (4 + (8 if raw else 0))
        gather += frames * 4 + 8 * 40 + (frames * 8 if ch.has_iq_outputs else 0) + (frames if cfg.flags & abi.FLAG_TRACE else 0)
    return {"ship_bytes_per_step": ship, "gather_bytes_per_step": gather}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_bench_split_device.json"))
    args = ap.parse_args()
    if args.steps < 20:
        raise SystemExit("--steps: time at least 20 steps")
    if args.warmup < 1:
        raise SystemExit("--warmup: at least one step (its outputs are the digest)")
    import torch
    from boondock_airband_b200 import configs, synth
    from boondock_airband_b200.engine import Engine

    n_gpus = torch.cuda.device_count()
    if n_gpus < 1:
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    K, W = args.steps, args.warmup
    base = configs.cfg4()
    base.max_batches_per_step = 8
    dev = base.devices[0]
    fs = dev.sample_rate
    hop_bytes = 8 * round(fs / base.wave_rate)
    step_bytes = 8 * fs  # one second of cf32 IQ
    lead = hop_bytes * 128 + 8 * base.fft_size  # the first step also fills the AGC look-back
    total = (K + W) * step_bytes + lead
    tmpl = synth.synth_torch(dev, int(TEMPLATE_S * fs), 0, torch.device("cuda", 0), gate_on=0.35, gate_off=0.12)
    reps = -(-total // (tmpl.numel() * 4))
    stream = tmpl.repeat(reps)[: total // 4].contiguous()
    del tmpl
    torch.cuda.synchronize()

    def arm(gpus=None, gpu_of_channel=None):
        cfg = configs.cfg4()
        cfg.max_batches_per_step = 8
        kw = {} if gpus is None else dict(gpus=gpus, gpu_of_channel=[gpu_of_channel])
        eng = Engine(cfg, **kw)
        assert eng.device_gpu(0) == 0
        eng.attach_device_stream(0, stream.data_ptr(), stream.numel() * 4)
        tickets, k1, k2 = [], [], []
        digest = hashlib.sha256()
        batches = [0]

        def retire(old, hashing):
            eng.ticket_ms(old)
            a, b = eng.kernel_ms(old)
            k1.append(a)
            k2.append(b)
            r = eng.collect_raw(old, 0)
            batches[0] += r.n_batches
            if hashing and r.n_batches:
                c, stride, w = r.channel_count, r.wave_stride, r.n_batches * r.wave_batch
                wave = C.string_at(r.waveout, 4 * c * stride)
                for ch in range(c):
                    digest.update(wave[4 * ch * stride: 4 * (ch * stride + w)])
                digest.update(C.string_at(r.status, 40 * r.n_batches * c))

        def run(n, first, hashing):
            for s in range(n):
                eng.advance_device_stream(0, step_bytes + (lead if (first and s == 0) else 0))
                tickets.append(eng.process())
                if len(tickets) >= DEPTH:
                    retire(tickets.pop(0), hashing)
            while tickets:
                retire(tickets.pop(0), hashing)

        run(W, True, True)
        k1.clear()
        k2.clear()
        batches[0] = 0
        t0 = time.perf_counter()
        run(K, False, False)
        wall = time.perf_counter() - t0
        launches = eng.launch_count()
        eng.close()
        assert batches[0] == K * 8, batches[0]
        out = {"gpus": gpus, "ms_per_step": 1e3 * wall / K, "x_realtime": K / wall,
               "k1_ms_per_step_max_over_members": statistics.median(k1), "k2_ms_per_step_max_over_members": statistics.median(k2),
               "launches": launches, "digest_of_warmup_outputs": digest.hexdigest()}
        out.update(traffic(cfg, gpu_of_channel))
        return out

    everything = [0] * 2000
    a, b = [], []
    for _ in range(args.reps):
        a.append(arm())
        b.append(arm([0], everything))
    c = arm([0, 0], [ch % 2 for ch in range(2000)])

    def summary(runs):
        ms = [r["ms_per_step"] for r in runs]
        return {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms), "ms_per_step_max": max(ms),
                "x_realtime_median": statistics.median(r["x_realtime"] for r in runs), "runs": runs}

    line = {"tool": "bench_split_device",
            "workload": "cfg4: 1 input, 61.44 Msps cf32, fft 8192, 2000 AM/NFM channels, device-resident IQ, audio to pinned host, 3 tickets in flight",
            "steps": K, "warmup": W, "reps": args.reps, **gpu_facts(),
            "a_plain_gpu0": summary(a), "b_split_over_0": summary(b), "c_split_over_0_0": c}
    if n_gpus >= 2:
        line["d_split_over_all"] = arm(list(range(n_gpus)), [ch % n_gpus for ch in range(2000)])
    else:
        line["d_split_over_all"] = "not measured: one GPU visible"
    digests = {r["digest_of_warmup_outputs"] for r in a + b + [c] + ([line["d_split_over_all"]] if n_gpus >= 2 else [])}
    line["outputs_equal_across_arms"] = len(digests) == 1
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
