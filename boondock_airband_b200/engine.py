"""Python host side of the engine: a thin ctypes binding of the C-ABI in include/ba_cuda.h.

``Engine`` plays the part of one ``demodulate()`` thread of the reference (boondock_airband.cpp:308-738) for the
devices in its ``EngineCfg``: input bytes go in with ``submit`` (the ``circbuffer_append`` of input-helpers.cpp:37-63),
``process`` runs one pass of the hot path over everything that is waiting, ``collect`` hands back what the reference
hands to its output thread after each batch (waveout, iq_out, axcindicate and the squelch levels).

All computation happens in libba_cuda.so (hand-written sm_100a kernels).  There is no fallback: if the library is
missing or no CUDA device is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

from . import abi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libba_cuda.so")

_LIBS = {}

# every symbol include/ba_cuda.h declares
SYMBOLS = (
    "ba_cuda_create", "ba_cuda_destroy", "ba_cuda_last_error", "ba_cuda_visible_devices", "ba_cuda_input_ring",
    "ba_cuda_submit", "ba_cuda_input_space", "ba_cuda_commit", "ba_cuda_input_consumed", "ba_cuda_submit_external", "ba_cuda_attach_device_stream",
    "ba_cuda_advance_device_stream", "ba_cuda_process", "ba_cuda_collect", "ba_cuda_collect_mixer", "ba_cuda_mixer_input_mask", "ba_cuda_set_freq_idx", "ba_cuda_ticket_ms", "ba_cuda_step_bytes",
    "ba_cuda_channel_info", "ba_cuda_window", "ba_cuda_debug_frames", "ba_cuda_debug_picks",
    "ba_cuda_debug_inject_picks", "ba_cuda_launch_count", "ba_cuda_kernel_ms", "ba_cuda_copy_ms", "ba_cuda_mark", "ba_cuda_mark_ms",
    "ba_cuda_create_multi", "ba_cuda_device_gpu", "ba_cuda_create_multi_split", "ba_cuda_channel_gpu",
)


class EngineError(RuntimeError):
    def __init__(self, where: str, code: int, text: str):
        super().__init__("%s: %s (%d) %s" % (where, abi.ERRORS.get(code, "?"), code, text))
        self.code = code


def load_library(path: Optional[str] = None):
    path = path or os.environ.get("BA_CUDA_LIB") or LIB_PATH  # BA_CUDA_LIB: tuning runs with an alternative build
    if path in _LIBS:
        return _LIBS[path]
    if not os.path.exists(path):
        raise FileNotFoundError(
            path + " is missing: build it with `make -C boondock_airband_b200/csrc` (or __graft_entry__.build()); "
            "there is no CPU implementation to fall back to")
    L = C.CDLL(path)
    vp, sz, u64p = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)
    L.ba_cuda_create.argtypes = [C.POINTER(abi.EngineDesc), C.POINTER(vp)]
    i32p = C.POINTER(C.c_int32)
    L.ba_cuda_create_multi.argtypes = [C.POINTER(abi.EngineDesc), i32p, C.c_int32, i32p, C.POINTER(vp)]
    L.ba_cuda_device_gpu.argtypes = [vp, C.c_int, i32p]
    L.ba_cuda_create_multi_split.argtypes = [C.POINTER(abi.EngineDesc), i32p, C.c_int32, i32p, C.POINTER(i32p), C.POINTER(vp)]
    L.ba_cuda_channel_gpu.argtypes = [vp, C.c_int, C.c_int, i32p]
    L.ba_cuda_destroy.argtypes = [vp]
    L.ba_cuda_destroy.restype = None
    L.ba_cuda_last_error.restype = C.c_char_p
    L.ba_cuda_visible_devices.argtypes = []
    L.ba_cuda_input_ring.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(sz), C.POINTER(sz)]
    L.ba_cuda_submit.argtypes = [vp, C.c_int, vp, sz]
    L.ba_cuda_commit.argtypes = [vp, C.c_int, sz]
    L.ba_cuda_submit_external.argtypes = [vp, C.c_int, vp, sz]
    L.ba_cuda_attach_device_stream.argtypes = [vp, C.c_int, vp, sz]
    L.ba_cuda_advance_device_stream.argtypes = [vp, C.c_int, sz]
    L.ba_cuda_process.argtypes = [vp]
    L.ba_cuda_collect.argtypes = [vp, C.c_int, C.c_int, C.POINTER(abi.StepOut)]
    L.ba_cuda_ticket_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    L.ba_cuda_step_bytes.argtypes = [vp, C.c_int, u64p, u64p]
    L.ba_cuda_channel_info.argtypes = [vp, C.c_int, C.c_int, C.POINTER(abi.ChannelInfo)]
    L.ba_cuda_window.argtypes = [vp, C.POINTER(C.c_float), sz]
    L.ba_cuda_debug_frames.argtypes = [vp, C.c_int, vp, sz, C.c_int, vp, vp]
    L.ba_cuda_debug_picks.argtypes = [vp, C.c_int, C.c_int, C.c_uint64, C.c_int, vp]
    L.ba_cuda_debug_inject_picks.argtypes = [vp, C.c_int, vp, C.c_int]
    L.ba_cuda_input_space.argtypes = [vp, C.c_int, C.POINTER(C.c_size_t)]
    L.ba_cuda_collect_mixer.argtypes = [vp, C.c_int, C.c_int, C.POINTER(abi.MixerOut)]
    L.ba_cuda_mixer_input_mask.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.ba_cuda_set_freq_idx.argtypes = [vp, C.c_int, C.c_int, C.c_int, u64p]
    L.ba_cuda_launch_count.argtypes = [vp, u64p]
    L.ba_cuda_kernel_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    L.ba_cuda_copy_ms.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    L.ba_cuda_mark.argtypes = [vp, C.c_int]
    L.ba_cuda_mark_ms.argtypes = [vp, C.c_int, C.c_int, C.POINTER(C.c_float)]
    _LIBS[path] = L
    return L


class StepResult:
    """What one ``process()`` produced for one device (views into pinned host memory, copied on access)."""

    def __init__(self, out: abi.StepOut):
        self.n_batches = out.n_batches
        self.wave_batch = out.wave_batch
        self.channel_count = out.channel_count
        self.frames_done = out.frames_done
        n = self.n_batches * self.wave_batch
        c, stride = self.channel_count, out.wave_stride
        self.rows_skipped = 0
        if n > 0:
            if out.waveout:
                full = np.ctypeslib.as_array(out.waveout, shape=(c, stride))
                self.waveout = full[:, :n].copy()
            else:
                # BA_FLAG_SKIP_SILENT_ROWS: only the rows that are not silence came back, plus where each one goes
                B = self.wave_batch
                self.waveout = np.zeros((c, n), np.float32)
                row_of = np.ctypeslib.as_array(out.row_of, shape=(c, out.row_of_stride))[:, :self.n_batches]
                rows = np.ctypeslib.as_array(out.rows, shape=(max(1, out.n_rows), B))
                for ch in range(c):
                    for b in range(self.n_batches):
                        r = int(row_of[ch, b])
                        if r >= 0:
                            assert r < out.n_rows
                            self.waveout[ch, b * B:(b + 1) * B] = rows[r]
                        else:
                            self.rows_skipped += 1
            self.iq_out = None
            if out.iq_out:
                iq = np.ctypeslib.as_array(out.iq_out, shape=(c, stride, 2))
                self.iq_out = iq[:, :n, :].copy()
            self.trace = None
            if out.trace:
                tr = np.ctypeslib.as_array(out.trace, shape=(c, stride))
                self.trace = tr[:, :n].copy()
            st = np.ctypeslib.as_array(C.cast(out.status, C.POINTER(C.c_uint32)), shape=(self.n_batches, c, 10)).copy()
            self.status_raw = st
        else:
            self.waveout = np.zeros((c, 0), np.float32)
            self.iq_out = None
            self.trace = None
            self.status_raw = np.zeros((0, c, 10), np.uint32)

    def status(self, batch: int, channel: int) -> dict:
        r = self.status_raw[batch, channel]
        f = r.view(np.float32)
        return dict(axcindicate=int(r[0].view(np.int32)), bin=int(r[1]), signal_level=float(f[2]), noise_level=float(f[3]),
                    squelch_level=float(f[4]), open_count=int(r[5]), flappy_count=int(r[6]), ctcss_count=int(r[7]),
                    no_ctcss_count=int(r[8]), active_counter=int(r[9]))


_CUDART = None


def device_to_host(ptr: int, nbytes: int) -> bytes:
    """cudaMemcpy of a device range to host bytes (for callers that asked for BA_FLAG_RESULTS_ON_DEVICE and want to look)."""
    global _CUDART
    if _CUDART is None:
        for name in ("libcudart.so", "libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
            try:
                _CUDART = C.CDLL(name)
                break
            except OSError:
                continue
        if _CUDART is None:
            raise RuntimeError("libcudart not found")
        _CUDART.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    buf = C.create_string_buffer(nbytes)
    rc = _CUDART.cudaMemcpy(buf, C.c_void_p(ptr), nbytes, 2)  # cudaMemcpyDeviceToHost
    if rc != 0:
        raise RuntimeError("cudaMemcpy -> %d" % rc)
    return buf.raw


class Engine:
    def __init__(self, cfg: abi.EngineCfg, lib_path: Optional[str] = None, gpus: Optional[Sequence[int]] = None,
                 gpu_of_device: Optional[Sequence[int]] = None, gpu_of_channel: Optional[Sequence[Optional[Sequence[int]]]] = None):
        """One engine on cfg.cuda_device; with ``gpus`` (CUDA ordinals, repeats allowed) one engine over those GPUs
        (ba_cuda_create_multi): devices are placed by ``gpu_of_device`` (indices into gpus) or, without it, with the
        devices of a mixer kept together and groups dealt out round robin.  ``gpu_of_channel`` (one entry per device:
        None, or per channel an index into gpus) spreads a device's channels over several GPUs
        (ba_cuda_create_multi_split): the device is channelized at its home, each channel demodulated where it is put.
        Every method works the same either way."""
        self.cfg = cfg
        self.L = load_library(lib_path)
        desc, self._keep = abi.build_desc(cfg)
        h = C.c_void_p()
        if gpus is None:
            if gpu_of_device is not None or gpu_of_channel is not None:
                raise ValueError("gpu_of_device and gpu_of_channel need gpus")
            rc = self.L.ba_cuda_create(C.byref(desc), C.byref(h))
            where = "ba_cuda_create"
        else:
            if gpu_of_device is not None and len(gpu_of_device) != len(cfg.devices):
                raise ValueError("gpu_of_device has %d entries for %d devices" % (len(gpu_of_device), len(cfg.devices)))
            g = (C.c_int32 * max(1, len(gpus)))(*gpus)
            m = None if gpu_of_device is None else (C.c_int32 * max(1, len(gpu_of_device)))(*gpu_of_device)
            if gpu_of_channel is None:
                rc = self.L.ba_cuda_create_multi(C.byref(desc), g, len(gpus), m, C.byref(h))
                where = "ba_cuda_create_multi"
            else:
                if len(gpu_of_channel) != len(cfg.devices):
                    raise ValueError("gpu_of_channel has %d entries for %d devices" % (len(gpu_of_channel), len(cfg.devices)))
                i32p = C.POINTER(C.c_int32)
                rows = [None if x is None else (C.c_int32 * max(1, len(x)))(*x) for x in gpu_of_channel]
                for x, dev in zip(gpu_of_channel, cfg.devices):
                    if x is not None and len(x) != len(dev.channels):
                        raise ValueError("gpu_of_channel entry has %d indices for %d channels" % (len(x), len(dev.channels)))
                table = (i32p * len(rows))(*[C.cast(r, i32p) if r is not None else i32p() for r in rows])
                self._keep = (self._keep, rows, table)
                rc = self.L.ba_cuda_create_multi_split(C.byref(desc), g, len(gpus), m, table, C.byref(h))
                where = "ba_cuda_create_multi_split"
        if rc != 0:
            raise EngineError(where, rc, self.L.ba_cuda_last_error().decode())
        self.h = h
        self._pins: List[object] = []

    def close(self):
        if getattr(self, "h", None):
            self.L.ba_cuda_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, where: str, rc: int) -> int:
        if rc < 0:
            raise EngineError(where, rc, self.L.ba_cuda_last_error().decode())
        return rc

    # ---- input side
    def submit(self, dev: int, iq: np.ndarray):
        """Append interleaved IQ to the device's pinned ring (circbuffer_append, input-helpers.cpp:37-63)."""
        iq = np.ascontiguousarray(iq)
        self._check("ba_cuda_submit", self.L.ba_cuda_submit(self.h, dev, iq.ctypes.data, iq.nbytes))

    def submit_external(self, dev: int, ptr: int, nbytes: int, keepalive=None):
        if keepalive is not None:
            self._pins.append(keepalive)
        self._check("ba_cuda_submit_external", self.L.ba_cuda_submit_external(self.h, dev, ptr, nbytes))

    def input_ring(self, dev: int):
        buf, size, mirror = C.c_void_p(), C.c_size_t(), C.c_size_t()
        self._check("ba_cuda_input_ring", self.L.ba_cuda_input_ring(self.h, dev, C.byref(buf), C.byref(size), C.byref(mirror)))
        return buf.value, size.value, mirror.value

    def input_space(self, dev: int) -> int:
        n = C.c_size_t()
        self._check("ba_cuda_input_space", self.L.ba_cuda_input_space(self.h, dev, C.byref(n)))
        return n.value

    def commit(self, dev: int, nbytes: int):
        self._check("ba_cuda_commit", self.L.ba_cuda_commit(self.h, dev, nbytes))

    def attach_device_stream(self, dev: int, device_ptr: int, capacity: int):
        self._check("ba_cuda_attach_device_stream", self.L.ba_cuda_attach_device_stream(self.h, dev, device_ptr, capacity))

    def advance_device_stream(self, dev: int, nbytes: int):
        self._check("ba_cuda_advance_device_stream", self.L.ba_cuda_advance_device_stream(self.h, dev, nbytes))

    # ---- one pass of the hot path
    def process(self) -> int:
        return self._check("ba_cuda_process", self.L.ba_cuda_process(self.h))

    def collect_raw(self, ticket: int, dev: int) -> abi.StepOut:
        out = abi.StepOut()
        self._check("ba_cuda_collect", self.L.ba_cuda_collect(self.h, ticket, dev, C.byref(out)))
        return out

    def collect(self, ticket: int, dev: int) -> StepResult:
        return StepResult(self.collect_raw(ticket, dev))

    def collect_mixer(self, ticket: int, mixer: int) -> dict:
        """What mixer_thread would hand on for this step: dict(first_batch, left [n], right [n] or None, axcindicate [n_batches])."""
        out = abi.MixerOut()
        self._check("ba_cuda_collect_mixer", self.L.ba_cuda_collect_mixer(self.h, ticket, mixer, C.byref(out)))
        n = out.n_batches * out.wave_batch
        left = np.ctypeslib.as_array(out.waveout, shape=(n,)).copy() if n else np.zeros(0, np.float32)
        right = None
        if out.stereo:
            right = np.ctypeslib.as_array(out.waveout_r, shape=(n,)).copy() if n else np.zeros(0, np.float32)
        sig = np.ctypeslib.as_array(out.axcindicate, shape=(out.n_batches,)).copy() if out.n_batches else np.zeros(0, np.int32)
        return dict(first_batch=int(out.first_batch), n_batches=int(out.n_batches), left=left, right=right, axcindicate=sig)

    def mixer_input_mask(self, mixer: int, input: int, enabled: bool):
        self._check("ba_cuda_mixer_input_mask", self.L.ba_cuda_mixer_input_mask(self.h, mixer, input, 1 if enabled else 0))

    def set_freq_idx(self, dev: int, channel: int, freq_idx: int) -> int:
        """Scan mode: switch the channel to freqlist[freq_idx] from the next process() on; returns the first batch it applies to."""
        b = C.c_uint64()
        self._check("ba_cuda_set_freq_idx", self.L.ba_cuda_set_freq_idx(self.h, dev, channel, freq_idx, C.byref(b)))
        return b.value

    def ticket_ms(self, ticket: int) -> float:
        ms = C.c_float()
        self._check("ba_cuda_ticket_ms", self.L.ba_cuda_ticket_ms(self.h, ticket, C.byref(ms)))
        return ms.value

    def copy_ms(self, ticket: int):
        """(host->device ms, device->host ms) of a finished ticket."""
        ms = (C.c_float * 2)()
        self._check("ba_cuda_copy_ms", self.L.ba_cuda_copy_ms(self.h, ticket, ms))
        return float(ms[0]), float(ms[1])

    def kernel_ms(self, ticket: int):
        ms = (C.c_float * 2)()
        self._check("ba_cuda_kernel_ms", self.L.ba_cuda_kernel_ms(self.h, ticket, ms))
        return ms[0], ms[1]

    def step_bytes(self, ticket: int):
        a, b = C.c_uint64(), C.c_uint64()
        self._check("ba_cuda_step_bytes", self.L.ba_cuda_step_bytes(self.h, ticket, C.byref(a), C.byref(b)))
        return a.value, b.value

    def mark(self, which: int):
        self._check("ba_cuda_mark", self.L.ba_cuda_mark(self.h, which))

    def mark_ms(self, a: int, b: int) -> float:
        ms = C.c_float()
        self._check("ba_cuda_mark_ms", self.L.ba_cuda_mark_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def device_gpu(self, dev: int) -> int:
        """CUDA ordinal that device ``dev`` runs on: where its device-resident stream and device results must live."""
        n = C.c_int32()
        self._check("ba_cuda_device_gpu", self.L.ba_cuda_device_gpu(self.h, dev, C.byref(n)))
        return n.value

    def channel_gpu(self, dev: int, ch: int) -> int:
        """CUDA ordinal whose demodulator runs channel ``ch`` of device ``dev`` (device_gpu(dev) unless the device is split)."""
        n = C.c_int32()
        self._check("ba_cuda_channel_gpu", self.L.ba_cuda_channel_gpu(self.h, dev, ch, C.byref(n)))
        return n.value

    def launch_count(self) -> int:
        n = C.c_uint64()
        self._check("ba_cuda_launch_count", self.L.ba_cuda_launch_count(self.h, C.byref(n)))
        return n.value

    # ---- inspection / parity hooks
    def channel_info(self, dev: int, ch: int) -> abi.ChannelInfo:
        info = abi.ChannelInfo()
        self._check("ba_cuda_channel_info", self.L.ba_cuda_channel_info(self.h, dev, ch, C.byref(info)))
        return info

    def window(self) -> np.ndarray:
        w = np.empty(self.cfg.fft_size, np.float32)
        self._check("ba_cuda_window", self.L.ba_cuda_window(self.h, w.ctypes.data_as(C.POINTER(C.c_float)), w.size))
        return w

    def debug_frames(self, dev: int, iq: np.ndarray, n_frames: int, want_in=True, want_out=True):
        iq = np.ascontiguousarray(iq)
        n = self.cfg.fft_size
        fi = np.empty((n_frames, n, 2), np.float32) if want_in else None
        fo = np.empty((n_frames, n, 2), np.float32) if want_out else None
        self._check("ba_cuda_debug_frames", self.L.ba_cuda_debug_frames(
            self.h, dev, iq.ctypes.data, iq.nbytes, n_frames, None if fi is None else fi.ctypes.data, None if fo is None else fo.ctypes.data))
        return fi, fo

    def debug_picks(self, dev: int, ch: int, first: int, count: int) -> np.ndarray:
        out = np.empty((count, 2), np.float32)
        self._check("ba_cuda_debug_picks", self.L.ba_cuda_debug_picks(self.h, dev, ch, first, count, out.ctypes.data))
        return out

    def inject_picks(self, dev: int, picks: np.ndarray):
        """picks: [n_frames][channels][2] float32 (test hook, see ba_cuda_debug_inject_picks)."""
        picks = np.ascontiguousarray(picks, np.float32)
        self._check("ba_cuda_debug_inject_picks", self.L.ba_cuda_debug_inject_picks(self.h, dev, picks.ctypes.data, picks.shape[0]))

    # ---- convenience: run a whole in-memory stream through the engine, as a file input would
    def run_stream(self, streams: List[np.ndarray], chunk_bytes: Optional[int] = None):
        """Feed streams[dev] (interleaved IQ arrays) in ring-sized chunks and return, per device, a dict with the
        concatenated waveout [C][n], iq_out, trace and the list of per-batch status rows."""
        nd = len(self.cfg.devices)
        views = [np.ascontiguousarray(s).view(np.uint8).reshape(-1) for s in streams]
        pos = [0] * nd
        acc = self._new_acc()
        if chunk_bytes is None:
            chunk_bytes = 1 << 20
        while True:
            fed = False
            for d in range(nd):
                if pos[d] < views[d].size:
                    # an input that a mixer holds back (it is ahead of the mixer's other inputs) stops draining its ring
                    n = min(chunk_bytes, views[d].size - pos[d], self.input_space(d))
                    if n > 0:
                        self.submit(d, views[d][pos[d]:pos[d] + n])
                        pos[d] += n
                        fed = True
            produced, advanced = self._step_into(acc)
            if not fed and not produced and not advanced:
                break
        return self._finish_acc(acc)

    def run_file_inputs(self, inputs, idle_sleep: float = 0.0002):
        """The demodulator side of a file replay: inputs[dev] is a started host.FileInput appending to device dev's ring
        from its own thread (file_rx_thread, input-file.cpp:82-147).  Runs until every input has hit end of file
        (state INPUT_FAILED, as in the reference) and the rings are drained; returns what run_stream returns."""
        import time
        acc = self._new_acc()
        while True:
            ended = all(i.state in (3, 4) for i in inputs)  # INPUT_FAILED / INPUT_STOPPED, read BEFORE the pass
            produced, advanced = self._step_into(acc)
            if ended and not produced and not advanced:
                break
            if not advanced:
                time.sleep(idle_sleep)  # demodulate() sleeps 10 ms here (boondock_airband.cpp:421-423)
        return self._finish_acc(acc)

    def _new_acc(self):
        self.mixed = [dict(left=[], right=[], axcindicate=[], next_batch=0) for _ in self.cfg.mixers]
        return [dict(waveout=[], iq_out=[], trace=[], status=[], frames_done=0) for _ in self.cfg.devices]

    def _step_into(self, acc):
        """One process() + collect() of every device; returns (some batch came out, some frame was consumed)."""
        t = self.process()
        produced = advanced = False
        for d in range(len(acc)):
            r = self.collect(t, d)
            advanced |= r.frames_done != acc[d]["frames_done"]
            acc[d]["frames_done"] = r.frames_done
            if r.n_batches:
                produced = True
                acc[d]["rows_skipped"] = acc[d].get("rows_skipped", 0) + r.rows_skipped
                acc[d]["waveout"].append(r.waveout)
                if r.iq_out is not None:
                    acc[d]["iq_out"].append(r.iq_out)
                if r.trace is not None:
                    acc[d]["trace"].append(r.trace)
                for b in range(r.n_batches):
                    acc[d]["status"].append([r.status(b, c) for c in range(r.channel_count)])
        for m, a in enumerate(self.mixed):
            r = self.collect_mixer(t, m)
            if r["n_batches"]:
                assert r["first_batch"] == a["next_batch"], (m, r["first_batch"], a["next_batch"])
                a["next_batch"] += r["n_batches"]
                a["left"].append(r["left"])
                if r["right"] is not None:
                    a["right"].append(r["right"])
                a["axcindicate"].append(r["axcindicate"])
                produced = True
        return produced, advanced

    def mixer_results(self):
        """After run_stream / run_file_inputs: per mixer dict(left, right or None, axcindicate)."""
        out = []
        for m, a in enumerate(self.mixed):
            cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt)
            out.append(dict(left=cat(a["left"], np.float32), right=cat(a["right"], np.float32) if self.cfg.mixers[m].stereo else None,
                            axcindicate=cat(a["axcindicate"], np.int32)))
        return out

    def _finish_acc(self, acc):
        out = []
        for d, a in enumerate(acc):
            c = len(self.cfg.devices[d].channels)
            out.append(dict(
                waveout=np.concatenate(a["waveout"], axis=1) if a["waveout"] else np.zeros((c, 0), np.float32),
                iq_out=np.concatenate(a["iq_out"], axis=1) if a["iq_out"] else None,
                trace=np.concatenate(a["trace"], axis=1) if a["trace"] else None,
                status=a["status"], frames_done=a["frames_done"], rows_skipped=a.get("rows_skipped", 0)))
        return out
