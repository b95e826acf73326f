#!/usr/bin/env python
"""bench.py — throughput of the channelize+demodulate hot path (BASELINE.json metric) on N B200s of one node.

Workload (config.workload): BASELINE.json configs[4], the box-scale multi-dongle sweep at its default point:
512 synthetic inputs x 2.56 Msps u8 IQ, fft_size 512, 16 AM channels each, WAVE_RATE 8000 — per GPU (weak scaling:
every rank runs its own 512 inputs; inputs share no state, so there is no collective on the data path).
A "step" is one pass of the hot path (ba_cuda_process) over one second of signal of every input
(8 WAVE_BATCH batches per channel): 512 x 2.56 M = 1310.72 M complex samples per GPU per step.

  value      every input's IQ already sits in HBM (its own buffer) when the timed region starts; the demodulated audio
             returns to pinned host memory inside the timed region (BASELINE.json: "only demodulated audio returns to host");
             value_results_on_device is the same run with the audio left in HBM for a consumer on the GPU
  e2e        the same steps through the C-ABI with HOST buffers: pinned host IQ -> H2D -> K1 -> K2 -> D2H of the audio
  roofline   dominant kernel (the channelizer) against the FP32 pipe (148 SMs x 128 lanes x 2 x 1.965 GHz, flops counted as
             5 N log2 N + 4 N + 4 C per frame) and against the measured HBM copy bandwidth (MEASURED_PEAKS.json; algorithmic
             bytes 2*b*Fs + 4*C*R per input-second, SURVEY.md section 8d)
  workloads  (N = 1) the other BASELINE.json configurations, device-resident, audio to the host: cfg1, cfg2, one GPU's share of
             cfg3, cfg4, cfg5 at fft 1024 / 2048 / 4096
  strong     (N > 1) cfg5 as BASELINE.json defines it: 512 inputs IN TOTAL, split i mod G over the G GPUs
  cpu_baseline / --impl reference
             the reference's CPU path (oracle/_ref: the reference's own squelch/ctcss/filters objects driven by the
             restated demodulate() loop, Release flags) on the host cores, one thread per input as the reference does
             with multiple_demod_threads, on a bounded sample of the same workload.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "aggregate IQ Msps channelized+demodulated per B200 (x real-time)"
FS = 2_560_000
WAVE_RATE = 8000
N_CHANNELS = 16
FFT_SIZE = 512
BATCHES_PER_STEP = 8  # one second of signal per input per step
TEMPLATES = 8         # distinct seeded streams; every input owns a private copy of one of them
DEPTH = 3             # tickets in flight (the engine has three result slots)
DUMP_ROWS = 1024      # (input, channel) rows --dump-outputs writes: 1024 x 8000 float32 samples = 32 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of each leg of the headline workload (the other workloads time 4 each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--inputs", type=int, default=512, help="inputs per GPU")
    ap.add_argument("--fft-size", type=int, default=FFT_SIZE)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-workloads", action="store_true")
    ap.add_argument("--total-inputs", type=int, default=512, help="inputs of the whole job in the strong-scaling leg (N > 1)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="signal seconds per input in the CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of `value` returned as DIR/*.npy (see dump_outputs)")
    return ap.parse_args()


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 10 ms while the GPU is under load
    (the same fields as the nvidia-smi line of B200_PROFILING.md; nvidia-smi -lms is too slow for a sub-second region)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as ex:  # noqa: BLE001
            self.err = repr(ex)
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((time.perf_counter(), sm, rs))
            except Exception as ex:  # noqa: BLE001
                self.err = repr(ex)
                return
            time.sleep(0.01)

    def stop(self, windows=None):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: %s" % self.err]}
        self.stop_flag.set()
        self.thread.join(timeout=2)
        nv = self.nv
        names = (("hw_slowdown", getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8)), ("hw_thermal_slowdown", getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                 ("sw_thermal_slowdown", getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)), ("sw_power_cap", getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)))
        rows = self.rows
        if windows:
            rows = [r for r in rows if any(a <= r[0] <= b for (a, b) in windows)]
        sm = [r[1] for r in rows]
        reasons = sorted({n for r in rows for (n, bit) in names if r[2] & bit})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_sm, "reasons": reasons, "samples": len(sm),
                "window": "timed regions (device-resident + end-to-end), NVML every 10 ms"}


def workload_cfg(n_inputs: int, fft_size: int, first_index: int, cuda_device: int):
    from boondock_airband_b200 import configs
    cfg = configs.cfg5(n_inputs, fft_size, first_index)
    cfg.cuda_device = cuda_device
    cfg.max_batches_per_step = BATCHES_PER_STEP
    return cfg


def dump_outputs(eng, ticket: int, n_inputs: int, out_dir: str):
    """What ba_cuda_collect returned for `ticket`, so that two builds can be compared output for output on the same seeded
    inputs.  Rows are (input, channel) pairs: all of them up to DUMP_ROWS, else a fixed seeded sample of DUMP_ROWS.
      rows.npy    [R, 2] float64   input and channel of each row
      audio.npy   [R, n] float32   the row's demodulated audio of the step (n = batches x WAVE_BATCH)
      status.npy  [R, batches, 10] float64   the row's per-batch status: axcindicate, bin, signal, noise and squelch level,
                                             open, flappy, ctcss and no-ctcss counts, active counter"""
    os.makedirs(out_dir, exist_ok=True)
    n_ch = len(eng.cfg.devices[0].channels)
    total = n_inputs * n_ch
    rows = np.arange(total) if total <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(total, DUMP_ROWS, replace=False))
    audio, status = [], []
    for i in np.unique(rows // n_ch):
        r = eng.collect(ticket, int(i))
        for c in rows[rows // n_ch == i] % n_ch:
            audio.append(r.waveout[c])
            raw = r.status_raw[:, c, :]
            st = raw.astype(np.float64)
            st[:, 0] = raw[:, 0].view(np.int32)
            st[:, 2:5] = raw[:, 2:5].view(np.float32)
            status.append(st)
    np.save(os.path.join(out_dir, "rows.npy"), np.stack([rows // n_ch, rows % n_ch], axis=1).astype(np.float64))
    np.save(os.path.join(out_dir, "audio.npy"), np.stack(audio).astype(np.float32))
    np.save(os.path.join(out_dir, "status.npy"), np.stack(status))


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference(n_inputs_total: int, fft_size: int, seconds: float, templates_host):
    """The reference's CPU path on the host cores: one demod thread per input, `threads` at a time."""
    from oracle import ba_oracle
    from oracle.ba_oracle import Oracle
    threads = host_threads()
    if ba_oracle.have_ref() and os.path.exists(ba_oracle.lib_path(ref=True, fast=True)):
        kind, ref = "reference", True
    else:
        kind, ref = "port", False
        if not os.path.exists(ba_oracle.lib_path(False, True)):
            ba_oracle.build(ref=False)
    n_inputs = max(1, min(n_inputs_total, threads))
    cfg = workload_cfg(n_inputs, fft_size, 0, 0)
    n_bytes = int(seconds * FS) * 2
    tiled = [np.resize(t, n_bytes) for t in templates_host]  # the templates repeat to cover `seconds`
    iqs = [tiled[i % len(tiled)] for i in range(n_inputs)]
    o = Oracle(cfg, ref=ref, keep=False, fast=True)
    # warm-up on a short prefix (page-in, FFT plan), then the timed pass on a fresh oracle
    o.run_threads([a[: n_bytes // 8] for a in iqs], threads)
    o.close()
    o = Oracle(cfg, ref=ref, keep=False, fast=True)
    wall = o.run_threads(iqs, threads)
    o.close()
    samples = n_inputs * (n_bytes // 2)
    msps = samples / wall / 1e6
    lanes = o.fft_lanes()
    fft_kind = ("in-repo AVX2+FMA radix-4 Stockham, eight consecutive frames per vector (oracle.cpp Fft8); the reference plans FFTW_MEASURE, FFTW is not installed on this box"
                if lanes == 8 else "in-repo scalar radix-4 Stockham (no AVX2 on this host)")
    out = {"value": msps, "unit": "Msps", "x_realtime": msps * 1e6 / FS, "cores": min(threads, n_inputs), "host_threads": threads, "kind": kind,
           "sample": "%d inputs x %.1f s of the same workload (cfg5: 2.56 Msps u8, fft %d, 16 AM channels), one thread per input, IQ fed from memory" % (n_inputs, seconds, fft_size),
           "fft_kind": fft_kind, "flags": "-O3 -ffast-math -march=x86-64-v3 (the binary travels to the GPU box), one translation unit instead of -flto",
           "wall_s": wall}
    try:
        out.update(fft_witness(fft_size, min(threads, n_inputs), FS // WAVE_RATE))
    except Exception as ex:  # noqa: BLE001
        out["fft_only_witness_note"] = repr(ex)
    return out


def fft_witness(fft_size: int, threads: int, hop: int):
    """What a tuned library FFT does on the same cores: torch.fft.fft (MKL / pocketfft) over a batch of complex64 frames, transform only -
    no sample conversion, window, bin pick or demodulation - expressed as the input rate it would sustain (frames/s x hop).  The CPU
    arm above does all of those; a reader can bound what FFTW would add or save from the two figures."""
    import torch
    before = torch.get_num_threads()
    torch.set_num_threads(threads)
    try:
        x = torch.randn(threads * 2048, fft_size, dtype=torch.complex64)
        torch.fft.fft(x, dim=1)
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            torch.fft.fft(x, dim=1)
        dt = (time.perf_counter() - t0) / reps
    finally:
        torch.set_num_threads(before)
    fps = x.shape[0] / dt
    return {"fft_only_witness_msps": fps * hop / 1e6, "fft_only_witness": "torch.fft.fft, complex64, batch %d x %d, %d threads: %.2f us per frame per thread" % (x.shape[0], fft_size, threads, 1e6 * threads / fps)}


def make_templates(seconds_total: float, device):
    """TEMPLATES distinct seeded input streams of seconds_total each, generated on `device` (torch is plumbing here)."""
    from boondock_airband_b200 import configs, synth
    cfg = configs.cfg5(TEMPLATES, FFT_SIZE, 0)
    n = int(round(seconds_total * FS))
    return [synth.synth_torch(cfg.devices[i], n, i, device) for i in range(TEMPLATES)]


def other_workloads(device):
    """The BASELINE.json configurations other than the headline one, measured inside this run (device-resident IQ, audio to
    pinned host memory; tools/bench_workloads.py holds the harness): Msps, x real time, K1 / K2 milliseconds per step."""
    import importlib.util

    import torch
    spec = importlib.util.spec_from_file_location("bench_workloads", os.path.join(ROOT, "tools", "bench_workloads.py"))
    bw = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bw)
    table = bw.workloads()
    out = {}
    for name in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5_n1024", "cfg5_n2048", "cfg5_n4096"):
        text, make = table[name]
        try:
            r = bw.run(name, text, make, 4, 2, device)
            out[name] = {"what": text, "msps": r["msps"], "x_realtime": r["x_realtime"], "x_realtime_aggregate": r["x_realtime_aggregate"], "ms_per_step": r["ms_per_step"],
                         "channelize_ms_per_step": r["channelize_ms_per_step"], "demod_ms_per_step": r["demod_ms_per_step"], "inputs": r["inputs"], "channels": r["channels"],
                         "fft_size": r["fft_size"], "steps": r["steps"], "warmup": r["warmup"]}
        except Exception as ex:  # noqa: BLE001
            out[name] = {"what": text, "error": repr(ex)}
        torch.cuda.empty_cache()
    return out


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version when the box sets
    NCCL_DEBUG): from here on file descriptor 1 is stderr, and emit() writes the result line to the real stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _RESULT_FD is None:
        os.write(1, data)
    else:
        os.write(_RESULT_FD, data)


def bind_near_gpu(local: int):
    """Run this rank on the CPUs next to its GPU (NVML's affinity mask) BEFORE pinned host memory is allocated, so that
    the rings and result buffers land on the GPU's NUMA node: with several ranks on one box the host<->device copies
    otherwise cross sockets and share one memory controller.  Returns the mask to restore for the CPU-baseline leg."""
    try:
        before = os.sched_getaffinity(0)
    except Exception:
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= before
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass
    return before


def main():
    args = parse_args()
    claim_stdout()
    rank, local, world = dist_env()
    if args.gpus != world and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE %d" % (args.gpus, world))
    K, W = args.steps, args.warmup
    step_samples = args.inputs * FS * BATCHES_PER_STEP * (WAVE_RATE // 8) // WAVE_RATE  # per GPU
    config = {"workload": "cfg5 box-scale multi-dongle: %d inputs x 2.56 Msps u8 per GPU, fft_size %d, %d AM channels/input, WAVE_RATE %d; "
                          "step = 1 s of signal per input (%d WAVE_BATCH batches)" % (args.inputs, args.fft_size, N_CHANNELS, WAVE_RATE, BATCHES_PER_STEP),
              "inputs_per_gpu": args.inputs, "sample_rate": FS, "sample_format": "u8", "fft_size": args.fft_size, "channels_per_input": N_CHANNELS,
              "wave_rate": WAVE_RATE, "samples_per_step_per_gpu": step_samples, "parallelism": "inputs sharded over GPUs, no collective",
              "l2": "inputs larger than L2 (%.2f GB of fresh IQ per step)" % (2 * step_samples / 1e9),
              "results": "value: IQ resident in HBM, audio copied to pinned host memory; value_skip_silent_rows: the same, (channel, batch) rows of exact zeros left out of the copy (BA_FLAG_SKIP_SILENT_ROWS); value_results_on_device: audio stays in HBM (BA_FLAG_RESULTS_ON_DEVICE), status returns to the host; e2e: host copies both ways"}

    import torch

    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes what the GPU path returned: it has no meaning with --impl reference")
        if rank != 0:
            return
        # bounded sample of the same workload on the host cores; templates are made with numpy-free torch CPU ops
        cpu_dev = torch.device("cpu")
        secs = args.cpu_seconds
        tmpl = [t.numpy() for t in make_templates(2.0, cpu_dev)]
        vals = []
        for _ in range(max(1, min(W, 1))):
            cpu_reference(args.inputs, args.fft_size, min(1.0, secs), tmpl)
        last = None
        for _ in range(K):
            last = cpu_reference(args.inputs, args.fft_size, secs, tmpl)
            vals.append(last["value"])
        v = statistics.median(vals)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Msps", "x_realtime": v * 1e6 / FS, "n_gpus": args.gpus, "steps": len(vals),
                "warmup": W, "ms_per_step": 1e3 * last["wall_s"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": "Msps", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
                "e2e": {"value": v, "unit": "Msps", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        emit(line)
        return

    from boondock_airband_b200.engine import Engine

    if args.dump_outputs and K < 1:
        raise SystemExit("--dump-outputs writes the last timed step: it needs --steps 1 or more")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    affinity_before = bind_near_gpu(local)
    total_steps = K + W
    step_bytes = 2 * FS * BATCHES_PER_STEP * (WAVE_RATE // 8) // WAVE_RATE  # bytes of one input per step (u8 IQ)
    # ---------------- device-resident run
    need = args.inputs * (total_steps + 0.05) * 2 * FS  # a private HBM copy of the whole timed stream per input
    free_b, _total_b = torch.cuda.mem_get_info(local)
    if need > 0.9 * free_b:
        raise SystemExit("--steps %d --warmup %d needs %.0f GB of device-resident IQ (%.0f GB free): lower --steps" % (K, W, need / 1e9, free_b / 1e9))
    tmpl = make_templates(total_steps + 0.05, device)
    from boondock_airband_b200 import sharding
    streams = []
    for i in range(args.inputs):
        streams.append(tmpl[i % TEMPLATES].clone())  # a private HBM copy per input
    lead = 2 * FS // WAVE_RATE * 128 + 2 * args.fft_size
    sampler = ClockSampler(local)
    sampler.start()
    windows = []

    def device_leg(flags, n_inputs=None, first_index=None, dump_dir=None):
        """K timed steps with the IQ resident in HBM; flags: where the results go (see the calls below); dump_dir: where
        dump_outputs writes what the last timed step returned."""
        n_in = args.inputs if n_inputs is None else n_inputs
        cfg = workload_cfg(n_in, args.fft_size, sharding.first_input_of_rank(args.inputs, rank) if first_index is None else first_index, local)
        cfg.flags = flags
        eng = Engine(cfg)
        for i, t in enumerate(streams[:n_in]):
            eng.attach_device_stream(i, t.data_ptr(), t.numel())
        torch.cuda.synchronize()
        # the first step also has to fill the AGC look-back (B + E frames): hand it a little more than one second
        tickets = []
        last = [None]

        copy_legs = [0.0, 0.0]
        d2h_total = [0]

        def run_steps(n, first):
            k1 = k2 = 0.0
            batches = 0
            for s in range(n):
                extra = lead if (first and s == 0) else 0
                for i in range(n_in):
                    eng.advance_device_stream(i, step_bytes + extra)
                t = eng.process()
                tickets.append(t)
                last[0] = t
                if len(tickets) >= DEPTH:
                    old = tickets.pop(0)
                    r = eng.collect_raw(old, 0)
                    a, b = eng.kernel_ms(old)
                    k1 += a
                    k2 += b
                    h, d = eng.copy_ms(old)
                    copy_legs[0] += h
                    copy_legs[1] += d
                    d2h_total[0] += eng.step_bytes(old)[1]
                    batches += r.n_batches
            while tickets:
                old = tickets.pop(0)
                r = eng.collect_raw(old, 0)
                a, b = eng.kernel_ms(old)
                k1 += a
                k2 += b
                h, d = eng.copy_ms(old)
                copy_legs[0] += h
                copy_legs[1] += d
                d2h_total[0] += eng.step_bytes(old)[1]
                batches += r.n_batches
            return k1, k2, batches

        run_steps(W, True)
        copy_legs[0] = copy_legs[1] = 0.0
        d2h_total[0] = 0
        launches0 = eng.launch_count()
        barrier()
        eng.mark(0)
        t0 = time.perf_counter()
        k1_ms, k2_ms, batches = run_steps(K, W == 0)
        eng.mark(1)
        barrier()
        t1 = time.perf_counter()
        wall = t1 - t0
        dev_ms = eng.mark_ms(0, 1)
        windows.append((t0, t1))
        launches = eng.launch_count() - launches0
        assert batches == K * BATCHES_PER_STEP, "device-resident run produced %d batches, expected %d" % (batches, K * BATCHES_PER_STEP)
        if dump_dir is not None:
            dump_outputs(eng, last[0], n_in, dump_dir)
        # timed on the device (CUDA events on the engine's own streams, behind the barrier), max over ranks; the host's wall clock
        # around the same region also contains the closing NCCL barrier and is reported next to it
        elapsed = dev_ms / 1e3
        if world > 1:
            elapsed = sharding.max_over_ranks(elapsed, dist, device)
            wall = sharding.max_over_ranks(wall, dist, device)
        eng.close()
        return {"elapsed": elapsed, "wall": wall, "dev_ms": dev_ms, "k1_ms": k1_ms, "k2_ms": k2_ms, "launches": launches, "copy_legs": list(copy_legs), "d2h_bytes": d2h_total[0]}

    # `value`: IQ resident in HBM, the demodulated audio copied to pinned host memory inside the timed region (the data flow
    # BASELINE.json names).  The same run with the results left in HBM for a consumer on the GPU (BA_FLAG_RESULTS_ON_DEVICE:
    # ba_cuda_collect hands out device pointers; per-batch status still returns to the host) is reported beside it as
    # `value_results_on_device`; the end-to-end leg below has host copies both ways.
    from boondock_airband_b200 import abi as _abi
    leg_dev = device_leg(_abi.FLAG_RESULTS_ON_DEVICE)
    leg_host = device_leg(0, dump_dir=args.dump_outputs if rank == 0 else None)
    # the same as `value`, but only the (channel, batch) rows that are not silence cross the link (BA_FLAG_SKIP_SILENT_ROWS: decided on
    # the data on the device; the synthetic carriers are keyed 1.5 s on / 0.5 s off, so about a quarter of the rows are silence)
    leg_skip = device_leg(_abi.FLAG_SKIP_SILENT_ROWS)
    elapsed, wall, dev_ms, k1_ms, k2_ms, launches, copy_legs = (leg_host[k] for k in ("elapsed", "wall", "dev_ms", "k1_ms", "k2_ms", "launches", "copy_legs"))
    # strong scaling (N > 1): BASELINE.json's cfg5 is 512 inputs in total; input i of the job runs on GPU i mod G
    strong = None
    if world > 1:
        mine = sharding.inputs_of_rank(args.total_inputs, world, rank)
        leg_strong = device_leg(0, n_inputs=len(mine), first_index=mine[0] if mine else 0)
        strong = {"total_inputs": args.total_inputs, "inputs_per_gpu": len(mine), "partition": "input i -> GPU i mod G", "ms_per_step": 1e3 * leg_strong["elapsed"] / K,
                  "value": args.total_inputs * FS * K / leg_strong["elapsed"] / 1e6, "unit": "Msps", "results": "audio copied to pinned host memory",
                  "kernels_ms_per_step": {"channelize(K1)": leg_strong["k1_ms"] / K, "demod(K2)": leg_strong["k2_ms"] / K}}
        strong["x_realtime"] = strong["value"] * 1e6 / FS
    del streams
    torch.cuda.empty_cache()

    # ---------------- end to end: pinned host IQ -> H2D -> kernels -> D2H audio, through the C-ABI
    e2e = None
    if not args.no_e2e:
        cfg2 = workload_cfg(args.inputs, args.fft_size, sharding.first_input_of_rank(args.inputs, rank), local)
        eng2 = Engine(cfg2)
        host = []
        for i in range(TEMPLATES):
            h = torch.empty(step_bytes + lead, dtype=torch.uint8).pin_memory()
            h.copy_(tmpl[i][: step_bytes + lead])
            host.append(h)
        # every input gets its own pinned buffer (no sharing of host pages between inputs)
        hbuf = [host[i % TEMPLATES].clone().pin_memory() if i >= TEMPLATES else host[i] for i in range(args.inputs)]
        torch.cuda.synchronize()
        h2d = d2h = 0
        pend = []
        e2e_legs = [0.0, 0.0, 0.0, 0.0]

        def e2e_note(old):
            a, b = eng2.copy_ms(old)
            c, d = eng2.kernel_ms(old)
            for i, v in enumerate((a, b, c, d)):
                e2e_legs[i] += v

        def e2e_steps(n, first):
            nonlocal h2d, d2h
            got = 0
            for s in range(n):
                nbytes = step_bytes + (lead if (first and s == 0) else 0)
                for i in range(args.inputs):
                    eng2.submit_external(i, hbuf[i].data_ptr(), nbytes)
                t = eng2.process()
                pend.append(t)
                if len(pend) >= DEPTH:
                    old = pend.pop(0)
                    r = eng2.collect_raw(old, args.inputs - 1)
                    got += r.n_batches
                    a, b = eng2.step_bytes(old)
                    h2d, d2h = h2d + a, d2h + b
                    e2e_note(old)
            while pend:
                old = pend.pop(0)
                r = eng2.collect_raw(old, args.inputs - 1)
                got += r.n_batches
                a, b = eng2.step_bytes(old)
                h2d, d2h = h2d + a, d2h + b
                e2e_note(old)
            return got

        e2e_steps(W, True)
        h2d = d2h = 0
        e2e_legs = [0.0, 0.0, 0.0, 0.0]
        barrier()
        t0 = time.perf_counter()
        got = e2e_steps(K, W == 0)
        barrier()
        e2e_wall = time.perf_counter() - t0
        windows.append((t0, t0 + e2e_wall))
        assert got == K * BATCHES_PER_STEP, "end-to-end run produced %d batches, expected %d" % (got, K * BATCHES_PER_STEP)
        if world > 1:
            e2e_wall = sharding.max_over_ranks(e2e_wall, dist, device)
        e2e_msps = sharding.aggregate_msps(world, K, step_samples, e2e_wall)
        e2e = {"value": e2e_msps, "unit": "Msps", "x_realtime": e2e_msps * 1e6 / FS, "h2d_bytes_per_step": h2d // K, "d2h_bytes_per_step": d2h // K,
               "ms_per_step": 1e3 * e2e_wall / K, "path": "ba_cuda_submit_external (pinned host) -> ba_cuda_process -> ba_cuda_collect",
               "legs_ms_per_step": {"h2d": e2e_legs[0] / K, "d2h": e2e_legs[1] / K, "channelize(K1)": e2e_legs[2] / K, "demod(K2)": e2e_legs[3] / K}}
        eng2.close()
        # the ceiling of this leg is the host link: time one large pinned host -> device copy on the same box
        try:
            probe_h = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
            probe_d = torch.empty(1 << 30, dtype=torch.uint8, device=device)
            probe_d.copy_(probe_h, non_blocking=True)
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(3):
                probe_d.copy_(probe_h, non_blocking=True)
            ev1.record()
            torch.cuda.synchronize()
            gbs = 3 * (1 << 30) / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
            e2e["host_link_h2d_gbs"] = gbs
            e2e["host_link_bound_msps"] = gbs * 1e9 / 2 / 1e6  # u8 IQ: 2 bytes per complex sample
            ev0.record()
            for _ in range(3):
                probe_h.copy_(probe_d, non_blocking=True)
            ev1.record()
            torch.cuda.synchronize()
            e2e["host_link_d2h_gbs"] = 3 * (1 << 30) / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
            del probe_h, probe_d
        except Exception as ex:  # noqa: BLE001
            e2e["host_link_h2d_gbs"] = None
            e2e["host_link_note"] = repr(ex)

    clocks = sampler.stop(windows)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = sharding.aggregate_msps(world, K, step_samples, elapsed)
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    algo_bytes_step = args.inputs * (2 * 1 * FS + 4 * N_CHANNELS * WAVE_RATE)  # per GPU per step (1 s of signal per input)
    # flops of the channelizer per frame, FFT convention: 5 N log2 N (butterflies) + 4 N (u8 conversion x window) + 4 C (magnitudes)
    n_fft = args.fft_size
    flops_frame = 5 * n_fft * (n_fft.bit_length() - 1) + 4 * n_fft + 4 * N_CHANNELS
    algo_flops_step = args.inputs * BATCHES_PER_STEP * (WAVE_RATE // 8) * flops_frame
    kern = {"channelize(K1)": k1_ms / K, "demod(K2)": k2_ms / K}
    legs = {"descriptors_h2d_ms": copy_legs[0] / K, "results_d2h_ms": copy_legs[1] / K}
    dom = "channelize(K1)"
    dom_ms = kern[dom]
    sm_count = torch.cuda.get_device_properties(local).multi_processor_count
    sm_ghz = float(peaks.get("sm_max_mhz", 1965.0)) / 1e3
    fp32_peak = sm_count * 128 * 2 * sm_ghz / 1e3  # TFLOP/s: 128 FP32 lanes per SM, one FMA = 2 flops
    achieved_tf = algo_flops_step / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
    achieved_gbs = algo_bytes_step / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum per launch of the same kernel, from the committed ncu --set full capture
    traffic, traffic_src, fma_busy = None, None, None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("inputs_per_gpu") == args.inputs and tj.get("fft_size") == args.fft_size:
            traffic, traffic_src = tj["dram_bytes_per_launch"].get(dom), tj.get("source")
            fma_busy = tj.get("fma_pipe_busy_pct")
    except Exception:
        pass
    roofline = {"bound": "fp32", "kernel": dom, "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved_tf / fp32_peak,
                "peak_source": "%d SMs x 128 FP32 lanes x 2 flops x %.3f GHz (no measured FP32 figure in MEASURED_PEAKS.json)" % (sm_count, sm_ghz),
                "flop_convention": "per frame 5 N log2 N + 4 N + 4 C = %d (N = %d, C = %d); the kernel's own operation count is lower (radix 16/32 butterflies)" % (flops_frame, n_fft, N_CHANNELS),
                "algorithmic_flops_per_launch": algo_flops_step, "frac_fp32": achieved_tf / fp32_peak,
                "hbm": {"achieved": achieved_gbs, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved_gbs / peak, "frac_of_spec_8000_gbs": achieved_gbs / 8000.0,
                        "algorithmic_bytes_per_launch": algo_bytes_step},
                "frac_hbm": achieved_gbs / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel_ms_per_launch": dom_ms,
                "all_kernels_ms_per_step": kern, "copy_legs_ms_per_step": legs, "fma_pipe_busy_pct_ncu": fma_busy,
                "note": "kernel times are event-bracketed on the kernels' own streams in the `value` leg (audio to the host): there K2 of a step is queued behind "
                        "K1 of the same step on one stream (plain-only large steps; ba_engine.cu), so K1 and K2 add up; in the results-on-device leg K2 of step t runs "
                        "beside K1 of step t+1 on a second stream (its figures: value_results_on_device_kernels_ms_per_step)"}
    value_dev = sharding.aggregate_msps(world, K, step_samples, leg_dev["elapsed"])
    line = {"metric": METRIC, "value": value, "unit": "Msps", "x_realtime": value * 1e6 / FS, "x_realtime_per_gpu": value * 1e6 / FS / world, "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * elapsed / K, "device_ms_per_step": dev_ms / K, "wall_ms_per_step": 1e3 * wall / K,
            "results_d2h_ms_per_step": copy_legs[1] / K,
            "value_results_on_device": value_dev, "ms_per_step_results_on_device": 1e3 * leg_dev["elapsed"] / K,
            "value_results_on_device_kernels_ms_per_step": {"channelize(K1)": leg_dev["k1_ms"] / K, "demod(K2)": leg_dev["k2_ms"] / K},
            "value_skip_silent_rows": sharding.aggregate_msps(world, K, step_samples, leg_skip["elapsed"]), "ms_per_step_skip_silent_rows": 1e3 * leg_skip["elapsed"] / K,
            "d2h_bytes_per_step": leg_host["d2h_bytes"] // K, "d2h_bytes_per_step_skip_silent_rows": leg_skip["d2h_bytes"] // K,
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (%d seeded streams, a private HBM copy per input)" % TEMPLATES, "config": config,
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline}
    if strong is not None:
        line["strong"] = strong
    if e2e is not None:
        line["e2e"] = e2e
    if world == 1 and not args.no_workloads:
        line["workloads"] = other_workloads(device)
    if world == 1 and not args.no_cpu:
        if affinity_before:
            os.sched_setaffinity(0, affinity_before)  # the CPU baseline gets every host thread
        tmpl_host = [t[: 2 * 2 * FS].cpu().numpy() for t in tmpl]
        line["cpu_baseline"] = {k: v for k, v in cpu_reference(args.inputs, args.fft_size, args.cpu_seconds, tmpl_host).items() if k != "wall_s"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
