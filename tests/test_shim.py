"""The drop-in boundary as a compiled artefact (SURVEY.md section 8b): boondock_airband_b200/csrc/demodulate_cuda.cpp, the
thread body that takes demodulate()'s place, built against include/ba_ref_layout.h and run between a fake rx thread
(circbuffer_append's arithmetic into the engine's pinned ring, under buffer_lock) and a fake output thread (output.cpp:931-951).
tests/shim/harness.cpp plays the reference's side; everything it calls in the product goes through the C-ABI."""
import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from boondock_airband_b200 import abi, configs, synth

import scenarios

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference/src"


@pytest.fixture(scope="module")
def shim():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "boondock_airband_b200", "csrc")], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", os.path.join(HERE, "shim")], stdout=subprocess.DEVNULL)
    libs = {}
    for name, rate in (("am", 8000), ("nfm", 16000)):
        L = C.CDLL(os.path.join(HERE, "shim", "libba_shim_%s_TESTONLY.so" % name))
        L.ba_shim_wave_rate.restype = C.c_int
        L.ba_shim_run.argtypes = [C.POINTER(abi.EngineDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t]
        L.ba_shim_run.restype = C.c_int
        L.ba_shim_batches.restype = C.c_long
        L.ba_shim_wave.argtypes = [C.c_int, C.c_int, C.POINTER(C.POINTER(C.c_float))]
        L.ba_shim_wave.restype = C.c_size_t
        L.ba_shim_axc.argtypes = [C.c_int, C.c_int, C.POINTER(C.POINTER(C.c_int))]
        L.ba_shim_axc.restype = C.c_size_t
        L.ba_shim_sizeof.argtypes = [C.c_int]
        L.ba_shim_sizeof.restype = C.c_size_t
        assert L.ba_shim_wave_rate() == rate
        libs[rate] = L
    return libs


PROBE = r"""
#include <cstdio>
#include <cstddef>
%s
int main() {
    printf("%%zu %%zu %%zu %%zu\n", sizeof(input_t), sizeof(freq_t), sizeof(channel_t), sizeof(device_t));
    printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu\n", offsetof(input_t, buf_size), offsetof(input_t, bufe), offsetof(input_t, state), offsetof(input_t, sfmt),
           offsetof(input_t, bytes_per_sample), offsetof(input_t, rx_thread), offsetof(input_t, buffer_lock));
    printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu\n", offsetof(freq_t, agcavgfast), offsetof(freq_t, ampfactor), offsetof(freq_t, squelch), offsetof(freq_t, active_counter),
           offsetof(freq_t, notch_filter), offsetof(freq_t, lowpass_filter), offsetof(freq_t, modulation));
    printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu\n", offsetof(channel_t, waveout), offsetof(channel_t, iq_in), offsetof(channel_t, iq_out), offsetof(channel_t, dm_dphi),
           offsetof(channel_t, axcindicate), offsetof(channel_t, afc), offsetof(channel_t, freqlist), offsetof(channel_t, freq_idx), offsetof(channel_t, has_iq_outputs),
           offsetof(channel_t, outputs));
    printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu\n", offsetof(device_t, channel_count), offsetof(device_t, bins), offsetof(device_t, channels), offsetof(device_t, waveend),
           offsetof(device_t, waveavail), offsetof(device_t, tag_queue), offsetof(device_t, mode), offsetof(device_t, output_overrun_count));
    return 0;
}
"""
STUBS = {
    "lame/lame.h": "typedef struct lame_global_struct* lame_t;\n",
    "shout/shout.h": "typedef struct shout shout_t;\n",
    "libconfig.h++": "namespace libconfig { class Setting; class Config; }\n",
    "fftw3.h": "typedef struct fftwf_plan_s* fftwf_plan; typedef float fftwf_complex[2];\n",
    "config.h": "/* what cmake would generate from config.h.in; nothing the structures depend on */\n",
}


@pytest.mark.parametrize("nfm", [False, True])
def test_layout_matches_the_reference_headers(nfm):
    """include/ba_ref_layout.h against the reference's own boondock_airband.h (compiled with stub headers in place of lame,
    shout, libconfig++ and fftw, which are not installed): sizes and the offsets of every member the thread body touches.
    tests/golden/ref_layout.json holds the probe's output for the reference's header (recorded from include/ba_ref_layout.h
    at a commit where this test had found the two equal), so the check runs without the reference tree; where the tree is
    mounted the probe also runs on the reference's header itself."""
    with open(os.path.join(HERE, "golden", "ref_layout.json")) as f:
        want = json.load(f)["nfm" if nfm else "am"]
    with tempfile.TemporaryDirectory() as td:
        for rel, text in STUBS.items():
            os.makedirs(os.path.dirname(os.path.join(td, "stubs", rel)), exist_ok=True)
            with open(os.path.join(td, "stubs", rel), "w") as f:
                f.write(text)
        probes = [("mine", '#include "ba_ref_layout.h"', ["-I" + os.path.join(ROOT, "include")])]
        if os.path.isdir(REF):
            probes.append(("ref", '#include "boondock_airband.h"', ["-I" + os.path.join(td, "stubs"), "-I" + REF]))
        for tag, inc, flags in probes:
            src = os.path.join(td, tag + ".cpp")
            with open(src, "w") as f:
                f.write(PROBE % inc)
            exe = os.path.join(td, tag)
            subprocess.check_call(["g++", "-std=c++14", "-w"] + (["-DNFM"] if nfm else []) + flags + [src, "-o", exe])
            got = subprocess.check_output([exe]).decode()
            assert got == want, "%s:\n%s---\nreference:\n%s" % (tag, got, want)


def test_shim_builds_and_loads_without_a_gpu(shim):
    for rate, L in shim.items():
        wave_len = 2 * (rate // 8) + 100
        assert L.ba_shim_sizeof(7) == 4 * wave_len  # offsetof(channel_t, waveout): wavein[WAVE_LEN] comes first


def bind(L):
    L.ba_shim_wave_rate.restype = C.c_int
    L.ba_shim_run.argtypes = [C.POINTER(abi.EngineDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t]
    L.ba_shim_run.restype = C.c_int
    L.ba_shim_wave.argtypes = [C.c_int, C.c_int, C.POINTER(C.POINTER(C.c_float))]
    L.ba_shim_wave.restype = C.c_size_t
    L.ba_shim_axc.argtypes = [C.c_int, C.c_int, C.POINTER(C.POINTER(C.c_int))]
    L.ba_shim_axc.restype = C.c_size_t
    return L


def run_shim(L, cfg, streams, chunk):
    desc, keep = abi.build_desc(cfg)
    views = [np.ascontiguousarray(s).view(np.uint8).reshape(-1) for s in streams]
    ptrs = (C.c_void_p * len(views))(*[v.ctypes.data for v in views])
    sizes = (C.c_size_t * len(views))(*[v.size for v in views])
    # the harness stops the threads once this many hand-offs have been taken (not after a quiet spell: a loaded box makes those)
    L.ba_shim_expect_batches.argtypes = [C.c_long]
    L.ba_shim_expect_batches(sum(cfg.batches_for(d, v.size) for d, v in enumerate(views)))
    rc = L.ba_shim_run(C.byref(desc), ptrs, sizes, chunk)
    assert rc == 0, rc
    out = []
    for d, dev in enumerate(cfg.devices):
        rows = []
        for c in range(len(dev.channels)):
            p = C.POINTER(C.c_float)()
            n = L.ba_shim_wave(d, c, C.byref(p))
            w = np.ctypeslib.as_array(p, shape=(n,)).copy() if n else np.zeros(0, np.float32)
            q = C.POINTER(C.c_int)()
            m = L.ba_shim_axc(d, c, C.byref(q))
            a = np.ctypeslib.as_array(q, shape=(m,)).copy() if m else np.zeros(0, np.int32)
            rows.append((w, a))
        out.append(rows)
    return out


def check_against_run_stream(cfg, streams, got, lib=None):
    from boondock_airband_b200.engine import Engine
    eng = Engine(cfg, lib) if lib is not None else Engine(cfg)
    want = eng.run_stream(streams, chunk_bytes=300_000)
    eng.close()
    B = cfg.wave_rate // 8
    for d, dev in enumerate(cfg.devices):
        nb = cfg.batches_for(d, np.ascontiguousarray(streams[d]).view(np.uint8).size)
        assert nb >= 3
        for c in range(len(dev.channels)):
            w, a = got[d][c]
            ref = want[d]["waveout"][c]
            assert len(w) == len(ref) == nb * B, (d, c, len(w), len(ref), nb * B)
            assert np.array_equal(w.view(np.uint32), ref.view(np.uint32)), (d, c)
            assert list(a) == [row[c]["axcindicate"] for row in want[d]["status"]]
        assert any((got[d][c][1] == abi.SIGNAL).any() for c in range(len(dev.channels)))


def test_emu_demodulate_cuda_thread_body(oracle_built):
    """The same harness over the thread-emulated engine (tests/emu): the host logic of the thread body and of the ring path
    (ba_cuda_input_ring / ba_cuda_commit / ba_cuda_input_consumed) on the CPU-only dev box."""
    import parity
    emu = parity.lib_for("emu")
    subprocess.check_call(["make", "-C", os.path.join(HERE, "shim"), "emu"], stdout=subprocess.DEVNULL)
    L = bind(C.CDLL(os.path.join(HERE, "shim", "libba_shim_am_emu_TESTONLY.so")))
    cfg = configs.cfg1()
    cfg.devices[0].channels = cfg.devices[0].channels[:3]
    cfg.flags = 0
    cfg.max_batches_per_step = 1
    streams = [synth.synth(cfg.devices[0], 0.55, 3, gate_on=0.2, gate_off=0.1)]
    got = run_shim(L, cfg, streams, 200_000)
    check_against_run_stream(cfg, streams, got, emu)


@pytest.mark.gpu
@pytest.mark.parametrize("which,chunk", [("cfg1", 262144), ("cfg1", 100_001), ("mixed", 65536), ("multi", 131072), ("cfg1_skip_silence", 200_000)])
def test_demodulate_cuda_between_a_fake_rx_thread_and_a_fake_output_thread(shim, which, chunk, monkeypatch):
    """The audio the fake output thread takes out of channel_t::waveout equals, bit for bit, what Engine.run_stream produces from
    the same bytes through ba_cuda_submit; so do the per-batch indicators."""
    from boondock_airband_b200.engine import Engine
    if which.startswith("cfg1"):
        cfg = configs.cfg1()
        streams = [synth.synth(cfg.devices[0], 2.2, 3, gate_on=0.4, gate_off=0.15)]
        if which.endswith("skip_silence"):
            monkeypatch.setenv("BA_CUDA_SKIP_SILENT_ROWS", "1")  # the thread body then asks for packed rows and writes silence itself
    elif which == "mixed":
        cfg, streams = scenarios.mixed_options(1.5, afc=False)
    else:
        cfg, streams = scenarios.multi_device(0.9)
    cfg.flags = 0
    cfg.max_batches_per_step = 1  # the reference's cadence: one hand-off per WAVE_BATCH
    got = run_shim(shim[cfg.wave_rate], cfg, streams, chunk)
    check_against_run_stream(cfg, streams, got)
