"""One engine over several GPUs (ba_cuda_create_multi): a group of ordinary engines behind one handle.

Each GPU runs the same kernels on its own devices, so a group must give, device for device and mixer for mixer, exactly
what one engine over the whole descriptor gives.  On the thread-emulated build the GPUs are emulated devices
(BA_EMU_DEVICES); on a B200 several members share GPU 0, and all visible GPUs are used where there are more."""
import collections
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from boondock_airband_b200 import abi, configs, synth
from boondock_airband_b200.abi import ChannelCfg, DeviceCfg, EngineCfg, MixerCfg, MixerInputCfg

import parity
import scenarios

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu(oracle_built):
    return parity.lib_for("emu")


@pytest.fixture(scope="module")
def cuda():
    return parity.lib_for("cuda")


def combined(seconds=0.3):
    """One descriptor out of four scenarios: multi_device's three inputs, mixers_on_multi_device's three inputs with its
    mono and stereo mixers, mixed_options' s16 input (NFM, low-pass, CTCSS, notch, AFC) and scan_mode's two inputs."""
    md, s_md = scenarios.multi_device(seconds)
    mx, s_mx = scenarios.mixers_on_multi_device(seconds)
    mo, s_mo = scenarios.mixed_options(seconds)
    sc, s_sc = scenarios.scan_mode(seconds)
    devices = md.devices + mx.devices + mo.devices + sc.devices
    mixers = [MixerCfg(m.name, [MixerInputCfg(i.device + 3, i.channel, i.ampfactor, i.balance) for i in m.inputs]) for m in mx.mixers[:2]]
    assert mixers[1].stereo and not mixers[0].stereo
    cfg = EngineCfg(fft_size=512, wave_rate=16000, devices=devices, flags=abi.FLAG_TRACE, max_batches_per_step=2, mixers=mixers)
    return cfg, s_md + s_mx + s_mo + s_sc


SCAN_DEV = 7  # scan_mode's scan input in combined()


def drive(e, cfg, streams, chunk, depth):
    """Feeds every input `chunk` bytes at a time and keeps up to `depth` tickets in flight (depth process() calls before the
    first collect).  Switches the scan channel before every step and masks one mixer input at a fixed step.  Returns everything the
    engine handed out, per ticket and concatenated."""
    nd, nm = len(cfg.devices), len(cfg.mixers)
    views = [np.ascontiguousarray(s).view(np.uint8).reshape(-1) for s in streams]
    pos = [0] * nd
    out = dict(steps=[], dev=[collections.defaultdict(list) for _ in range(nd)], mix=[collections.defaultdict(list) for _ in range(nm)],
               switches=[])
    pending = collections.deque()
    quiet = step = 0

    def collect_one():
        t = pending.popleft()
        moved = False
        row = []
        for d in range(nd):
            r = e.collect(t, d)
            acc = out["dev"][d]
            moved |= r.n_batches > 0 or (acc["frames"] and acc["frames"][-1] != r.frames_done) or (not acc["frames"] and r.frames_done > 0)
            acc["frames"].append(r.frames_done)
            row.append((r.n_batches, r.frames_done))
            if r.n_batches:
                acc["waveout"].append(r.waveout)
                acc["status"].append(r.status_raw)
                if r.iq_out is not None:
                    acc["iq_out"].append(r.iq_out)
                if r.trace is not None:
                    acc["trace"].append(r.trace)
        for m in range(nm):
            r = e.collect_mixer(t, m)
            row.append((r["first_batch"], r["n_batches"]))
            if r["n_batches"]:
                moved = True
                a = out["mix"][m]
                a["left"].append(r["left"])
                if r["right"] is not None:
                    a["right"].append(r["right"])
                a["axcindicate"].append(r["axcindicate"])
                a["first_batch"].append(r["first_batch"])
        out["steps"].append(row)
        return moved

    while True:
        fed = False
        for d in range(nd):
            if pos[d] < views[d].size:
                n = min(chunk, views[d].size - pos[d], e.input_space(d))
                if n > 0:
                    e.submit(d, views[d][pos[d]:pos[d] + n])
                    pos[d] += n
                    fed = True
        out["switches"].append(e.set_freq_idx(SCAN_DEV, 0, step % 3))  # the scan channel moves through its list
        if step == 5 and nm:
            e.mixer_input_mask(0, 1, False)
        pending.append(e.process())
        step += 1
        if len(pending) >= depth:
            moved = collect_one()
            quiet = 0 if (moved or fed) else quiet + 1
            if quiet > depth + 1 and all(p == v.size for p, v in zip(pos, views)):
                break
    while pending:
        collect_one()
    out["consumed"] = [input_consumed(e, d) for d in range(nd)]
    return out


def input_consumed(e, dev):
    n = C.c_size_t()
    assert e.L.ba_cuda_input_consumed(e.h, C.c_int(dev), C.byref(n)) == 0
    return n.value


def assert_same(a, b, cfg):
    assert a["steps"] == b["steps"]
    assert a["switches"] == b["switches"]
    assert a["consumed"] == b["consumed"]
    for d in range(len(cfg.devices)):
        x, y = a["dev"][d], b["dev"][d]
        assert x["frames"] == y["frames"] and x["frames"][-1] > 0, d
        assert len(x["waveout"]) > 0, d
        for key in ("waveout", "iq_out", "trace", "status"):
            assert len(x[key]) == len(y[key]), (d, key)
            for p, q in zip(x[key], y[key]):
                assert p.shape == q.shape and np.array_equal(np.ascontiguousarray(p).view(np.uint8), np.ascontiguousarray(q).view(np.uint8)), (d, key)
    for m in range(len(cfg.mixers)):
        x, y = a["mix"][m], b["mix"][m]
        assert len(x["left"]) > 0 and x["first_batch"] == y["first_batch"], m
        for key in ("left", "right", "axcindicate"):
            assert len(x[key]) == len(y[key]), (m, key)
            for p, q in zip(x[key], y[key]):
                assert np.array_equal(p.view(np.uint32), q.view(np.uint32)), (m, key)


def run_group_against_one(lib, gpus, maps, chunk, depth, seconds=0.3):
    from boondock_airband_b200.engine import Engine
    cfg, streams = combined(seconds)
    e = Engine(cfg, lib)
    try:
        want = drive(e, cfg, streams, chunk, depth)
    finally:
        e.close()
    assert len(set(want["switches"])) >= 3 and sum(len(x["left"]) for x in want["mix"]) > 0
    for gmap in maps:
        g = Engine(cfg, lib, gpus=gpus, gpu_of_device=gmap)
        try:
            placed = [g.device_gpu(d) for d in range(len(cfg.devices))]
            got = drive(g, cfg, streams, chunk, depth)
            launches = g.launch_count()
        finally:
            g.close()
        assert launches > 0
        if gmap is not None:
            assert placed == [gpus[k] for k in gmap]
        assert_same(got, want, cfg)


@pytest.mark.parametrize("chunk,depth", [(300_000, 1), (777_777, 3)])
def test_emu_group_equals_one_engine(emu, monkeypatch, chunk, depth):
    """The combined descriptor over three emulated GPUs, with the default placement and with an explicit map, against one
    engine: every device's audio, iq_out, trace, status, frames and ring position, every mixer's planes, indicators and
    batch numbers, bit for bit.  Scan switches and a mixer input mask land at the same batches on both."""
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    run_group_against_one(emu, [0, 1, 2], [None, [2, 2, 1, 1, 1, 1, 0, 0, 2]], chunk, depth)


def small_cfg(n_devices=6, mixers=((1, 3), (3, 4))):
    devs = [DeviceCfg(sample_rate=2_560_000, centerfreq=120_000_000, channels=[ChannelCfg(freq=120_000_000 + 100_000 * (k - 1)) for k in range(2)])
            for _ in range(n_devices)]
    mx = [MixerCfg("m%d" % i, [MixerInputCfg(d, 0) for d in ins]) for i, ins in enumerate(mixers)]
    return EngineCfg(fft_size=512, wave_rate=8000, devices=devs, mixers=mx, max_batches_per_step=2)


def test_emu_placement(emu, monkeypatch):
    """Default placement keeps devices joined by mixers (transitively) together and deals groups out round robin in the
    order of their first device; an explicit map is followed; every bad argument is refused with its reason."""
    from boondock_airband_b200.engine import Engine, EngineError
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg = small_cfg()  # groups {0}, {1, 3, 4}, {2}, {5}
    e = Engine(cfg, emu, gpus=[2, 0, 1])
    assert [e.device_gpu(d) for d in range(6)] == [2, 0, 1, 0, 0, 2]
    e.close()
    e = Engine(small_cfg(mixers=()), emu, gpus=[1, 2])  # no mixers: device i -> gpus[i % n]
    assert [e.device_gpu(d) for d in range(6)] == [1, 2, 1, 2, 1, 2]
    e.close()
    e = Engine(cfg, emu, gpus=[0, 1, 2], gpu_of_device=[1, 2, 2, 2, 2, 0])
    assert [e.device_gpu(d) for d in range(6)] == [1, 2, 2, 2, 2, 0]
    with pytest.raises(EngineError, match="BAD_ARG.*no device 6"):
        e.device_gpu(6)
    e.close()
    plain_cfg = small_cfg()
    plain_cfg.cuda_device = 2
    e = Engine(plain_cfg, emu)
    assert [e.device_gpu(d) for d in range(6)] == [2] * 6
    e.close()
    refusals = [
        (dict(gpus=[]), "n_gpus 0"),
        (dict(gpus=[0, 3]), r"gpus\[1\] = 3 is not a visible CUDA device \(3 visible\)"),
        (dict(gpus=[0, -1]), r"gpus\[1\] = -1 is not a visible"),
        (dict(gpus=[0, 1, 2], gpu_of_device=[0, 0, 0, 0, 0, 3]), r"gpu_of_device\[5\] = 3 is not an index into the 3 gpus"),
        (dict(gpus=[0, 1, 2], gpu_of_device=[0, -1, 0, 0, 0, 0]), r"gpu_of_device\[1\] = -1"),
        (dict(gpus=[0, 1], gpu_of_device=[0, 1, 0, 1, 0, 0]), r"mixer 1 has inputs on gpus\[1\] and gpus\[0\]"),
        (dict(gpus=[0, 1], gpu_of_device=[0, 0, 0, 1, 1, 0]), r"mixer 0 has inputs on gpus\[0\] and gpus\[1\]"),
    ]
    for kw, msg in refusals:
        with pytest.raises(EngineError, match=msg) as ei:
            Engine(cfg, emu, **kw)
        assert ei.value.code == -4, kw  # BA_ERR_BAD_ARG


def test_emu_gpu_without_devices(emu, monkeypatch):
    """A GPU that receives no device gets no member; the group still runs and matches one engine."""
    from boondock_airband_b200.engine import Engine
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, streams = scenarios.multi_device(0.4)
    one = Engine(cfg, emu)
    want = one.run_stream(streams, chunk_bytes=300_000)
    one.close()
    for kw in (dict(gpus=[0, 1, 2, 1, 0]), dict(gpus=[0, 1, 2], gpu_of_device=[2, 0, 2])):
        g = Engine(cfg, emu, **kw)
        got = g.run_stream(streams, chunk_bytes=300_000)
        g.close()
        for d in range(3):
            assert got[d]["frames_done"] == want[d]["frames_done"] > 0
            assert np.array_equal(got[d]["waveout"].view(np.uint32), want[d]["waveout"].view(np.uint32))
            assert np.array_equal(got[d]["trace"], want[d]["trace"])
            assert got[d]["status"] == want[d]["status"]


def test_emu_group_skip_silent_rows(emu, monkeypatch):
    """BA_FLAG_SKIP_SILENT_ROWS over a group: each device's packed rows come from the member that holds it; put back
    together they are one engine's audio, bit for bit."""
    from boondock_airband_b200.engine import Engine
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, streams = scenarios.multi_device(0.5)
    cfg.flags = 0
    one = Engine(cfg, emu)
    want = one.run_stream(streams, chunk_bytes=300_000)
    one.close()
    cfg.flags = abi.FLAG_SKIP_SILENT_ROWS
    g = Engine(cfg, emu, gpus=[0, 1], gpu_of_device=[0, 1, 1])
    got = g.run_stream(streams, chunk_bytes=250_001)
    g.close()
    assert sum(got[d]["rows_skipped"] for d in range(3)) > 0
    for d in range(3):
        assert got[d]["waveout"].shape == want[d]["waveout"].shape
        assert np.array_equal(got[d]["waveout"].view(np.uint32), want[d]["waveout"].view(np.uint32)), d
        assert got[d]["status"] == want[d]["status"]


def test_emu_two_members_on_one_gpu_keep_their_shared_memory(emu, monkeypatch):
    """Two members on one GPU, the one with fewer channels (less K1 shared memory) created second.  The kernel's dynamic
    shared-memory limit is per (device, function): had the second member lowered it, the first member's next channelizer
    launch would be refused (the emulation refuses a launch above the limit set on its device)."""
    from boondock_airband_b200.engine import Engine
    monkeypatch.setenv("BA_EMU_DEVICES", "1")
    big = DeviceCfg(sample_rate=2_560_000, centerfreq=120_000_000, channels=[ChannelCfg(freq=120_000_000 + 60_000 * (k - 6)) for k in range(12)])
    small = DeviceCfg(sample_rate=2_560_000, centerfreq=121_000_000, channels=[ChannelCfg(freq=121_000_000 + 100_000 * k) for k in range(2)])
    cfg = EngineCfg(fft_size=512, wave_rate=8000, devices=[big, small], max_batches_per_step=2)
    streams = [synth.synth(d, 0.45, 60 + i, gate_on=0.2, gate_off=0.07) for i, d in enumerate(cfg.devices)]
    one = Engine(cfg, emu)
    want = one.run_stream(streams, chunk_bytes=300_000)
    one.close()
    g = Engine(cfg, emu, gpus=[0, 0], gpu_of_device=[0, 1])
    got = g.run_stream(streams, chunk_bytes=300_000)
    g.close()
    for d in range(2):
        assert got[d]["frames_done"] == want[d]["frames_done"] > 0
        assert got[d]["waveout"].shape[1] >= 2 * cfg.wave_batch
        assert np.array_equal(got[d]["waveout"].view(np.uint32), want[d]["waveout"].view(np.uint32))


def test_emu_drop_in_thread_body_over_two_gpus(emu, monkeypatch):
    """demodulate_cuda.cpp with BA_CUDA_DEVICES=0,1: the one demodulator thread of all devices spreads them over both GPUs
    as one engine; what the fake output thread takes is what Engine.run_stream gives."""
    from test_shim import bind, check_against_run_stream, run_shim
    monkeypatch.setenv("BA_EMU_DEVICES", "2")
    monkeypatch.setenv("BA_CUDA_DEVICES", "0,1")
    subprocess.check_call(["make", "-C", os.path.join(HERE, "shim"), "emu"], stdout=subprocess.DEVNULL)
    L = bind(C.CDLL(os.path.join(HERE, "shim", "libba_shim_am_emu_TESTONLY.so")))
    cfg, streams = scenarios.multi_device(0.5)
    cfg.flags = 0
    cfg.max_batches_per_step = 1
    got = run_shim(L, cfg, streams, 150_000)
    check_against_run_stream(cfg, streams, got, emu)


# ---------------------------------------------------------------------------------------------------------------- B200
def visible_gpus():
    from boondock_airband_b200 import engine as eng_mod
    return int(eng_mod.load_library().ba_cuda_visible_devices())


@pytest.mark.gpu
def test_group_equals_one_engine_on_gpu(cuda):
    """The combined descriptor over [0, 0, 0] (three members on one GPU) and, where there are several GPUs, over all of
    them: bit-identical to one engine, with three tickets in flight."""
    run_group_against_one(cuda, [0, 0, 0], [None, [2, 2, 1, 1, 1, 1, 0, 0, 2]], 777_777, 3, seconds=0.8)
    n = visible_gpus()
    if n >= 2:
        run_group_against_one(cuda, list(range(n)), [None], 300_000, 1, seconds=0.8)


@pytest.mark.gpu
def test_cfg5_full_size_over_two_members(cuda):
    """BASELINE cfg 5 at full size (512 inputs, 8192 plain AM channels, device-resident) over [0, 0]: every input's audio
    and status equal one engine's.  Each stream is allocated on the GPU device_gpu() names."""
    torch = pytest.importorskip("torch")
    from boondock_airband_b200.engine import Engine
    cfg = configs.cfg5(512, 512)
    cfg.max_batches_per_step = 4
    tmpl = [synth.synth(cfg.devices[k], 1.0, k, gate_on=0.35, gate_off=0.12) for k in range(8)]
    total = tmpl[0].size

    def run(**kw):
        e = Engine(cfg, cuda, **kw)
        keep, waves, stats = [], [[] for _ in range(512)], [[] for _ in range(512)]
        try:
            for i in range(512):
                t = torch.from_numpy(tmpl[i % 8].copy()).to(torch.device("cuda", e.device_gpu(i)))
                keep.append(t)
                e.attach_device_stream(i, t.data_ptr(), t.numel())
            for lo in range(0, total, 1_500_000):
                n = min(1_500_000, total - lo)
                for i in range(512):
                    e.advance_device_stream(i, n)
                while True:
                    tk = e.process()
                    got = 0
                    for i in range(512):
                        r = e.collect(tk, i)
                        if r.n_batches:
                            got += 1
                            waves[i].append(r.waveout)
                            stats[i].append(r.status_raw)
                    if not got:
                        break
        finally:
            e.close()
        return [np.concatenate(w, axis=1) for w in waves], [np.concatenate(s, axis=0) for s in stats]

    want_w, want_s = run()
    got_w, got_s = run(gpus=[0, 0])
    assert want_w[0].shape[1] // cfg.wave_batch == cfg.batches_for(0, total) >= 7
    for i in range(512):
        assert np.array_equal(got_w[i].view(np.uint32), want_w[i].view(np.uint32)), i
        assert np.array_equal(got_s[i], want_s[i]), i


@pytest.mark.gpu
def test_results_on_device_over_two_members(cuda):
    """BA_FLAG_RESULTS_ON_DEVICE over [0, 0]: the device pointers of each member hold what host results give."""
    from boondock_airband_b200.engine import Engine, device_to_host
    cfg, streams = scenarios.multi_device(0.6)
    cfg.flags = 0
    e = Engine(cfg, cuda, gpus=[0, 0])
    want = e.run_stream(streams, chunk_bytes=400_000)
    e.close()
    cfg.flags = abi.FLAG_RESULTS_ON_DEVICE
    e = Engine(cfg, cuda, gpus=[0, 0])
    waves = [[] for _ in cfg.devices]
    try:
        for lo in range(0, max(s.size for s in streams), 400_000):
            for d, s in enumerate(streams):
                if lo < s.size:
                    e.submit(d, s[lo:lo + 400_000])
            while True:
                t = e.process()
                got = 0
                for d in range(len(cfg.devices)):
                    out = e.collect_raw(t, d)
                    if out.n_batches:
                        got += 1
                        n = out.n_batches * out.wave_batch
                        base = C.cast(out.waveout, C.c_void_p).value
                        waves[d].append(np.stack([np.frombuffer(device_to_host(base + 4 * c * out.wave_stride, 4 * n), np.float32)
                                                  for c in range(out.channel_count)]))
                if not got:
                    break
    finally:
        e.close()
    for d in range(len(cfg.devices)):
        got = np.concatenate(waves[d], axis=1)
        assert got.shape == want[d]["waveout"].shape and got.shape[1] > 0
        assert np.array_equal(got.view(np.uint32), want[d]["waveout"].view(np.uint32)), d


@pytest.mark.gpu
def test_drop_in_thread_body_over_two_members(monkeypatch):
    """The shim's "multi" case with BA_CUDA_DEVICES=0,0: the thread body makes one engine of two members on GPU 0."""
    from test_shim import bind, check_against_run_stream, run_shim
    monkeypatch.setenv("BA_CUDA_DEVICES", "0,0")
    subprocess.check_call(["make", "-C", os.path.join(os.path.dirname(HERE), "boondock_airband_b200", "csrc")], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", os.path.join(HERE, "shim")], stdout=subprocess.DEVNULL)
    cfg, streams = scenarios.multi_device(0.9)
    cfg.flags = 0
    cfg.max_batches_per_step = 1
    L = bind(C.CDLL(os.path.join(HERE, "shim", "libba_shim_%s_TESTONLY.so" % ("am" if cfg.wave_rate == 8000 else "nfm"))))
    got = run_shim(L, cfg, streams, 131072)
    check_against_run_stream(cfg, streams, got)
