"""One engine over several GPUs (ba_cuda_create_multi) against plain engines, on the cfg5 workload of bench.py.

Inputs: configs.cfg5 (2.56 Msps u8, fft 512, 16 AM channels each), one private device-resident copy of a seeded stream per
input, allocated on the GPU the engine names for it (device_gpu).  Audio is copied to the engine's pinned host memory.
One step is one second of signal per input; three tickets are kept in flight as in bench.py.

Legs, each `--steps` timed steps after `--warmup` steps, (a) and (b) alternated `--reps` times in the same process:
  (a) a plain engine, 512 inputs on GPU 0
  (b) create_multi over [0], the same 512 inputs (the group only forwards calls)
  (c) create_multi over [0, 0], 256 inputs on each member
  (d) with G >= 2 visible GPUs: create_multi over all of them, 512 inputs per GPU, against G x (a)
Host cost: the host time of one ba_cuda_process() of a plain cfg5 engine, over calls made with fewer than three tickets
outstanding (they do not wait), and of one ba_cuda_collect() of a ticket that has finished (it does not wait either); both
through ctypes, so they include the binding's own call overhead.

Prints one JSON line.  Usage: python tools/bench_multi_gpu.py [--steps 20] [--warmup 3] [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

FS = 2_560_000
WAVE_RATE = 8000
FFT_SIZE = 512
BATCHES_PER_STEP = 8  # one second of signal per input per step
TEMPLATES = 8
DEPTH = 3
INPUTS = 512


def gpu_facts():
    import torch
    facts = {"gpu": torch.cuda.get_device_name(0), "visible_gpus": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        facts["power_limit_and_max_sm_clock"] = [ln.strip() for ln in q.stdout.strip().splitlines()]
    except (OSError, subprocess.SubprocessError) as ex:
        facts["power_limit_and_max_sm_clock"] = "not read: %s" % ex
    return facts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if args.steps < 20:
        raise SystemExit("--steps: time at least 20 steps")
    import torch
    from boondock_airband_b200 import configs, synth
    from boondock_airband_b200.engine import Engine

    n_gpus = torch.cuda.device_count()
    if n_gpus < 1:
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    K, W = args.steps, args.warmup
    total_s = K + W + 0.05
    step_bytes = 2 * FS  # one second of u8 IQ
    lead = 2 * FS // WAVE_RATE * 128 + 2 * FFT_SIZE  # the first step also fills the AGC look-back
    n_bytes = int(round(total_s * FS)) * 2

    # one private copy per input per GPU it may run on
    streams = {}
    for g in range(n_gpus if n_gpus >= 2 else 1):
        dev = torch.device("cuda", g)
        tcfg = configs.cfg5(TEMPLATES, FFT_SIZE, 0)
        tmpl = [synth.synth_torch(tcfg.devices[i], n_bytes // 2, i, dev) for i in range(TEMPLATES)]
        streams[g] = [tmpl[i % TEMPLATES].clone() for i in range(INPUTS)]
        del tmpl
    torch.cuda.synchronize()

    def leg(n_inputs, gpus=None, host_cost=False):
        cfg = configs.cfg5(n_inputs, FFT_SIZE, 0)
        cfg.max_batches_per_step = BATCHES_PER_STEP
        eng = Engine(cfg, gpus=gpus)
        used = {}
        for i in range(n_inputs):
            g = eng.device_gpu(i)
            k = used.get(g, 0)
            used[g] = k + 1
            t = streams[g][k]
            eng.attach_device_stream(i, t.data_ptr(), t.numel())
        tickets = []
        proc_us, coll_us = [], []
        batches = [0]

        def retire(old):
            eng.ticket_ms(old)  # waits for the ticket on every member
            if host_cost:
                for i in range(n_inputs):
                    t0 = time.perf_counter()
                    r = eng.collect_raw(old, i)
                    coll_us.append(1e6 * (time.perf_counter() - t0))
                    if i == 0:
                        batches[0] += r.n_batches
            else:
                batches[0] += eng.collect_raw(old, 0).n_batches

        def run(n, first):
            for s in range(n):
                extra = lead if (first and s == 0) else 0
                for i in range(n_inputs):
                    eng.advance_device_stream(i, step_bytes + extra)
                outstanding = len(tickets)
                t0 = time.perf_counter()
                t = eng.process()
                dt = time.perf_counter() - t0
                if outstanding < DEPTH:
                    proc_us.append(1e6 * dt)
                tickets.append(t)
                if len(tickets) >= DEPTH:
                    retire(tickets.pop(0))
            while tickets:
                retire(tickets.pop(0))

        run(W, True)
        proc_us.clear()
        coll_us.clear()
        batches[0] = 0
        eng.mark(0)
        t0 = time.perf_counter()
        run(K, W == 0)
        eng.mark(1)
        wall = time.perf_counter() - t0
        dev_ms = eng.mark_ms(0, 1)
        eng.close()
        assert batches[0] == K * BATCHES_PER_STEP, batches[0]
        out = {"inputs": n_inputs, "gpus": gpus, "ms_per_step": 1e3 * wall / K, "device_ms_per_step": dev_ms / K,
               "msps": n_inputs * FS * K / wall / 1e6, "x_realtime": n_inputs * K / wall}
        if host_cost:
            out["process_us_median"] = statistics.median(proc_us)
            out["process_calls"] = len(proc_us)
            out["collect_us_median"] = statistics.median(coll_us)
            out["collect_calls"] = len(coll_us)
        return out

    a, b = [], []
    for _ in range(args.reps):
        a.append(leg(INPUTS))
        b.append(leg(INPUTS, gpus=[0]))
    c = leg(INPUTS, gpus=[0, 0])
    host = leg(INPUTS, host_cost=True)

    def summary(runs):
        ms = [r["ms_per_step"] for r in runs]
        return {"ms_per_step_median": statistics.median(ms), "ms_per_step_min": min(ms), "ms_per_step_max": max(ms),
                "msps_median": statistics.median(r["msps"] for r in runs), "runs": runs}

    line = {"tool": "bench_multi_gpu", "workload": "cfg5 %d inputs x 2.56 Msps u8, fft %d, 16 AM channels, device-resident IQ, audio to pinned host" % (INPUTS, FFT_SIZE),
            "steps": K, "warmup": W, "reps": args.reps, **gpu_facts(),
            "a_plain_gpu0": summary(a), "b_multi_over_0": summary(b), "c_multi_over_0_0": c,
            "host_cost_plain_cfg5": {k: host[k] for k in ("process_us_median", "process_calls", "collect_us_median", "collect_calls", "ms_per_step")}}
    if n_gpus >= 2:
        d = leg(INPUTS * n_gpus, gpus=list(range(n_gpus)))
        a_med = statistics.median(r["msps"] for r in a)
        line["d_multi_over_all"] = dict(d, vs_G_times_a=d["msps"] / (n_gpus * a_med))
    else:
        line["d_multi_over_all"] = "not measured: one GPU visible"
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
