"""One input's channels demodulated on several GPUs (ba_cuda_create_multi_split): channelize once at the input's home,
demodulate everywhere, gather the results at home.

K2 is bit-exact given the same picks, and a bin's pick does not depend on which other bins are picked, so a split group
must give exactly what one plain engine gives on the same descriptor fed the same bytes in the same chunks.  On the
thread-emulated build the GPUs are emulated devices (BA_EMU_DEVICES); on a B200 the members share GPU 0 (real events
across members, peer stores that are same-device stores), and all visible GPUs are used where there are two or more."""
import collections
import ctypes as C
import hashlib

import numpy as np
import pytest

from boondock_airband_b200 import abi, configs, synth
from boondock_airband_b200.abi import ChannelCfg, DeviceCfg, EngineCfg, FreqCfg, MixerCfg, MixerInputCfg

import parity


@pytest.fixture(scope="module")
def emu(oracle_built):
    return parity.lib_for("emu")


@pytest.fixture(scope="module")
def cuda():
    return parity.lib_for("cuda")


def wideband(n_channels, sample_rate, fmt, centerfreq, iq_every=4):
    """A reduced cfg 4 input: AM plain and NFM with low-pass (every fourth NFM with CTCSS and notch); some channels
    with iq_out."""
    dev = configs.cfg4(n_channels=n_channels, sample_rate=sample_rate).devices[0]
    dev.sample_format = fmt
    shift = centerfreq - dev.centerfreq
    dev.centerfreq = centerfreq
    for i, c in enumerate(dev.channels):
        c.freq += shift
        c.has_iq_outputs = i % iq_every == 3
    return dev


def scenario(seconds=0.55, flags=abi.FLAG_TRACE):
    """Input A (cf32, 12 channels) and input B (s16, 9 channels) are split; input C (u8, AFC) is not.  A stereo mixer takes
    channel 0 of A (demodulated at A's home) and channel 1 of A (demodulated elsewhere)."""
    a = wideband(12, 2_048_000, "f32", 140_000_000)
    b = wideband(9, 2_400_000, "s16", 150_000_000)
    c = DeviceCfg(sample_rate=2_560_000, centerfreq=120_000_000, sample_format="u8",
                  channels=[ChannelCfg(freq=120_000_000 - 300_000 + 3_000, afc=8), ChannelCfg(freq=120_000_000 + 200_000)])
    mix = MixerCfg("ab", [MixerInputCfg(0, 0, 0.9, -0.4), MixerInputCfg(0, 1, 1.2, 0.5)])
    # a ring far larger than a chunk: what is fed never depends on when the copies of earlier tickets finished
    cfg = EngineCfg(fft_size=2048, wave_rate=16000, devices=[a, b, c], flags=flags, max_batches_per_step=1, mixers=[mix], ring_bytes=64 << 20)
    streams = [synth.synth(d, seconds, 70 + i, gate_on=0.25, gate_off=0.1) for i, d in enumerate(cfg.devices)]
    return cfg, streams


GPU_OF_DEVICE = [0, 1, 2]  # A at home on gpus[0], B on gpus[1], C on gpus[2]


def split_map(cfg):
    """A's channels go c % 3; B's even channels run on gpus[0], away from B's home (gpus[1] runs A's too: circular)."""
    return [[c % 3 for c in range(len(cfg.devices[0].channels))], [0 if c % 2 == 0 else 1 for c in range(len(cfg.devices[1].channels))], None]


def drive(e, cfg, streams, chunks, depth, inject=None):
    """Feeds input d `chunks[d]` bytes at a time (uneven across inputs) with up to `depth` tickets in flight; returns every
    result per device and mixer.  inject: {dev: picks [frames][channels][2]} fed through the pick-injection hook instead
    of bytes, one batch worth of frames per step."""
    nd, nm = len(cfg.devices), len(cfg.mixers)
    views = [np.ascontiguousarray(s).view(np.uint8).reshape(-1) for s in streams]
    pos = [0] * nd
    inj_pos = {d: 0 for d in (inject or {})}
    out = dict(dev=[collections.defaultdict(list) for _ in range(nd)], mix=[collections.defaultdict(list) for _ in range(nm)])
    pending = collections.deque()

    def collect_one():
        t = pending.popleft()
        moved = False
        for d in range(nd):
            r = e.collect(t, d)
            acc = out["dev"][d]
            moved = moved or r.n_batches > 0 or bool(acc["frames"] and acc["frames"][-1] != r.frames_done)
            acc["frames"].append(r.frames_done)
            if r.n_batches:
                for key in ("waveout", "status_raw", "iq_out", "trace"):
                    v = getattr(r, key)
                    if v is not None:
                        acc[key].append(v)
                acc["skipped"].append(r.rows_skipped)
        for m in range(nm):
            r = e.collect_mixer(t, m)
            if r["n_batches"]:
                moved = True
                for key in ("left", "right", "axcindicate", "first_batch"):
                    out["mix"][m][key].append(r[key])
        return moved

    quiet = 0
    while True:
        fed = False
        for d in range(nd):
            if inject and d in inject:
                p = inject[d]
                n = min(cfg.wave_batch, p.shape[0] - inj_pos[d])
                if n > 0:
                    e.inject_picks(d, p[inj_pos[d]:inj_pos[d] + n])
                    inj_pos[d] += n
                    fed = True
            elif pos[d] < views[d].size:
                n = min(chunks[d], views[d].size - pos[d])
                assert e.input_space(d) >= n, d  # the feed is the same on every engine, whatever the timing
                if n > 0:
                    e.submit(d, views[d][pos[d]:pos[d] + n])
                    pos[d] += n
                    fed = True
        pending.append(e.process())
        if len(pending) >= depth:
            moved = collect_one()
            quiet = 0 if (moved or fed) else quiet + 1
            if quiet > depth + 1:
                break
    while pending:
        collect_one()
    return out


def assert_same(a, b, cfg, keys=("waveout", "status_raw", "iq_out", "trace")):
    for d in range(len(cfg.devices)):
        x, y = a["dev"][d], b["dev"][d]
        assert x["frames"] == y["frames"] and x["frames"][-1] > 0, d
        assert len(x["waveout"]) >= 2, d
        for key in keys:
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


def plain_and_split(lib, gpus, depth, flags=abi.FLAG_TRACE, chunks=(1_300_007, 500_003, 400_001), seconds=0.55, inject=None):
    from boondock_airband_b200.engine import Engine
    cfg, streams = scenario(seconds, flags)
    one = Engine(cfg, lib)
    try:
        want = drive(one, cfg, streams, chunks, depth, inject)
    finally:
        one.close()
    g = Engine(cfg, lib, gpus=gpus, gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=split_map(cfg))
    try:
        placed = [[g.channel_gpu(d, c) for c in range(len(dev.channels))] for d, dev in enumerate(cfg.devices)]
        got = drive(g, cfg, streams, chunks, depth, inject)
    finally:
        g.close()
    gmap = split_map(cfg)
    for d, dev in enumerate(cfg.devices):
        home = gpus[GPU_OF_DEVICE[d]]
        assert placed[d] == [home if gmap[d] is None else gpus[gmap[d][c]] for c in range(len(dev.channels))], d
    return cfg, want, got


@pytest.mark.parametrize("depth", [1, 3])
def test_emu_split_equals_one_engine(emu, monkeypatch, depth):
    """The main scenario over three emulated GPUs, with one and three tickets in flight and uneven chunks: audio, iq_out,
    trace, status and frames of every input and the stereo mixer's planes and indicators, bit for bit."""
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, want, got = plain_and_split(emu, [0, 1, 2], depth)
    assert sum(len(x) for x in want["dev"][0]["iq_out"]) > 0
    assert_same(got, want, cfg)


def test_emu_split_skip_silent_rows(emu, monkeypatch):
    """BA_FLAG_SKIP_SILENT_ROWS: the home packs the gathered rows with its own; expanded, they are one engine's audio."""
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, want, got = plain_and_split(emu, [0, 1, 2], 3, flags=abi.FLAG_SKIP_SILENT_ROWS, seconds=0.7)
    assert sum(sum(x["skipped"]) for x in got["dev"]) > 0
    assert_same(got, want, cfg, keys=("waveout", "status_raw", "iq_out"))


def test_emu_split_keep_picks(emu, monkeypatch):
    """BA_FLAG_KEEP_PICKS ships every channel's picked IQ; debug_picks of a channel demodulated away from home reads the
    home's ring and equals one engine's."""
    from boondock_airband_b200.engine import Engine
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, streams = scenario(0.4, abi.FLAG_TRACE | abi.FLAG_KEEP_PICKS)
    res = []
    for kw in (dict(), dict(gpus=[0, 1, 2], gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=split_map(cfg))):
        e = Engine(cfg, emu, **kw)
        try:
            out = drive(e, cfg, streams, (1_000_003, 700_001, 500_009), 1)
            n = out["dev"][0]["frames"][-1]
            first = max(0, n - 600)
            res.append((out, [e.debug_picks(0, 1, first, n - first), e.debug_picks(1, 0, first, n - first), e.debug_picks(0, 5, first, n - first)]))
        finally:
            e.close()
    assert_same(res[1][0], res[0][0], cfg)
    for p, q in zip(res[1][1], res[0][1]):
        assert np.abs(p).max() > 0 and np.array_equal(p.view(np.uint32), q.view(np.uint32))


def test_emu_split_injected_picks(emu, monkeypatch):
    """Picks injected at the home of a split input reach the followers' shadows: the same outputs as one engine fed the
    same picks (input C keeps streaming bytes)."""
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    rng = np.random.default_rng(5)
    cfg, _ = scenario(0.1)
    inject = {}
    for d in (0, 1):
        nch = len(cfg.devices[d].channels)
        frames = 3 * cfg.wave_batch + 150
        env = (np.arange(frames) // 1500 % 2).astype(np.float32)[:, None, None]
        inject[d] = (rng.standard_normal((frames, nch, 2)).astype(np.float32) * 0.02 + 0.3 * env).astype(np.float32)
    cfg, want, got = plain_and_split(emu, [0, 1, 2], 1, inject=inject, seconds=0.45)
    assert_same(got, want, cfg)


def test_emu_no_split(emu, monkeypatch):
    """An all-home gpu_of_channel and NULL entries give the same outputs and the same launch count as ba_cuda_create_multi."""
    from boondock_airband_b200.engine import Engine
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, streams = scenario(0.35)
    chunks = (900_001, 600_007, 300_001)
    runs = []
    for gpc in (None, [[0] * len(cfg.devices[0].channels), None, [2] * len(cfg.devices[2].channels)], [None, None, None]):
        e = Engine(cfg, emu, gpus=[0, 1, 2], gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=gpc)
        try:
            runs.append((drive(e, cfg, streams, chunks, 3), e.launch_count()))
        finally:
            e.close()
    for out, launches in runs[1:]:
        assert launches == runs[0][1] > 0
        assert_same(out, runs[0][0], cfg)


def test_emu_split_placement_and_refusals(emu, monkeypatch):
    """channel_gpu and device_gpu follow the maps; every new refusal returns BA_ERR_BAD_ARG with its reason, the missing
    peer access one through the emulation's knob."""
    from boondock_airband_b200.engine import Engine, EngineError
    monkeypatch.setenv("BA_EMU_DEVICES", "3")
    cfg, _ = scenario(0.1)
    gmap = split_map(cfg)
    e = Engine(cfg, emu, gpus=[2, 0, 1], gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=gmap)
    assert [e.device_gpu(d) for d in range(3)] == [2, 0, 1]
    assert [e.channel_gpu(0, c) for c in range(12)] == [[2, 0, 1][c % 3] for c in range(12)]
    assert [e.channel_gpu(1, c) for c in range(9)] == [2 if c % 2 == 0 else 0 for c in range(9)]
    assert [e.channel_gpu(2, c) for c in range(2)] == [1, 1]
    assert e.channel_info(0, 4).bin == Engine(cfg, emu).channel_info(0, 4).bin
    with pytest.raises(EngineError, match="BAD_ARG.*device 0 has no channel 12"):
        e.channel_gpu(0, 12)
    e.close()
    plain = Engine(cfg, emu)
    assert plain.channel_gpu(1, 3) == plain.device_gpu(1) == 0
    plain.close()
    n0, n1 = len(cfg.devices[0].channels), len(cfg.devices[1].channels)
    refusals = [
        (dict(gpu_of_channel=[[0] * (n0 - 1) + [3], None, None]), r"gpu_of_channel\[0\]\[11\] = 3 is not an index into the 3 gpus"),
        (dict(gpu_of_channel=[None, [-1] + [1] * (n1 - 1), None]), r"gpu_of_channel\[1\]\[0\] = -1"),
        (dict(gpu_of_channel=[None, None, [2, 0]]), r"device 2 cannot be split: channel 0 has AFC"),
    ]
    for kw, msg in refusals:
        with pytest.raises(EngineError, match=msg) as ei:
            Engine(cfg, emu, gpus=[0, 1, 2], gpu_of_device=GPU_OF_DEVICE, **kw)
        assert ei.value.code == -4, kw
    monkeypatch.setenv("BA_EMU_NO_PEER", "1")
    with pytest.raises(EngineError, match=r"device 0 channel 1: GPU 1 and its home GPU 0 have no peer access") as ei:
        Engine(cfg, emu, gpus=[0, 1, 2], gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=gmap)
    assert ei.value.code == -4
    # two members on one ordinal need no peer access
    Engine(cfg, emu, gpus=[0, 0, 2], gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=[[c % 2 for c in range(n0)], None, None]).close()


def test_emu_remote_scan_channel(emu, monkeypatch):
    """set_freq_idx reaches a scan channel demodulated away from its home: a one-channel scan device whose only channel
    runs on the other GPU switches at the same batches, with the same audio, as on one engine."""
    from boondock_airband_b200.engine import Engine
    monkeypatch.setenv("BA_EMU_DEVICES", "2")
    fs, f0 = 2_560_000, 121_500_000
    scan = ChannelCfg(freq=f0, modulation="nfm", freqs=[FreqCfg(f0), FreqCfg(f0 + 25_000, modulation="nfm", bandwidth=12_500, ctcss=100.0),
                                                      FreqCfg(f0 + 50_000, squelch_threshold=-48, ampfactor=1.6)])
    dev = DeviceCfg(sample_rate=fs, centerfreq=f0 + 20 * (fs // 512), sample_format="u8", channels=[scan])
    cfg = EngineCfg(fft_size=512, wave_rate=16000, devices=[dev], flags=abi.FLAG_TRACE, max_batches_per_step=1)
    iq = synth.synth(dev, 0.9, 44, gate_on=0.22, gate_off=0.09)
    res = []
    for kw in (dict(), dict(gpus=[0, 1], gpu_of_device=[0], gpu_of_channel=[[1]])):
        e = Engine(cfg, emu, **kw)
        try:
            if kw:
                assert e.device_gpu(0) == 0 and e.channel_gpu(0, 0) == 1
            waves, switches, step = [], [], 0
            for lo in range(0, iq.size, 300_000):
                e.submit(0, iq[lo:lo + 300_000])
                while True:
                    switches.append(e.set_freq_idx(0, 0, step % 3))
                    step += 1
                    r = e.collect(e.process(), 0)
                    if not r.n_batches:
                        break
                    waves.append((r.waveout, r.trace, r.status_raw))
            res.append((waves, switches))
        finally:
            e.close()
    assert res[0][1] == res[1][1] and len(set(res[0][1])) >= 3 and len(res[0][0]) >= 4
    for (a, b) in zip(res[0][0], res[1][0]):
        for p, q in zip(a, b):
            assert np.array_equal(np.ascontiguousarray(p).view(np.uint8), np.ascontiguousarray(q).view(np.uint8))


# ---------------------------------------------------------------------------------------------------------------- B200
def visible_gpus():
    from boondock_airband_b200 import engine as eng_mod
    return int(eng_mod.load_library().ba_cuda_visible_devices())


@pytest.mark.gpu
def test_split_equals_one_engine_on_gpu(cuda):
    """The main scenario over [0, 0, 0]: three members on GPU 0, real events between them, with three tickets in flight."""
    cfg, want, got = plain_and_split(cuda, [0, 0, 0], 3, seconds=0.9)
    assert_same(got, want, cfg)


_CFG4_IQ = {}


def run_cfg4(lib, seconds, gpus=None, gpu_of_channel=None, flags=0):
    """Full-size cfg 4 (61.44 Msps cf32, fft 8192, 2000 channels, every 50th with iq_out) from a device-resident stream;
    per step a digest of every result (audio, status, iq_out), in order."""
    import torch
    from boondock_airband_b200.engine import Engine, device_to_host
    cfg = configs.cfg4()
    for i, c in enumerate(cfg.devices[0].channels):
        c.has_iq_outputs = i % 50 == 7
    cfg.max_batches_per_step = 4
    cfg.flags = flags
    dev = cfg.devices[0]
    n = int(seconds * dev.sample_rate)
    kw = {} if gpus is None else dict(gpus=gpus, gpu_of_channel=[gpu_of_channel])
    e = Engine(cfg, lib, **kw)
    digests = []
    try:
        key = (n, e.device_gpu(0))
        if key not in _CFG4_IQ:
            _CFG4_IQ[key] = synth.synth_torch(dev, n, 4, torch.device("cuda", key[1]), gate_on=0.35, gate_off=0.12)
            torch.cuda.synchronize()
        iq = _CFG4_IQ[key]
        e.attach_device_stream(0, iq.data_ptr(), iq.numel() * 4)
        step_bytes = 8 * dev.sample_rate // 4
        for lo in range(0, iq.numel() * 4, step_bytes):
            e.advance_device_stream(0, min(step_bytes, iq.numel() * 4 - lo))
            while True:
                t = e.process()
                r = e.collect_raw(t, 0)
                if not r.n_batches:
                    break
                h = hashlib.sha256()
                nb, c, stride, w = r.n_batches, r.channel_count, r.wave_stride, r.n_batches * r.wave_batch
                if flags & abi.FLAG_RESULTS_ON_DEVICE:
                    base = C.cast(r.waveout, C.c_void_p).value
                    wave = np.frombuffer(device_to_host(base, 4 * c * stride), np.float32).reshape(c, stride)[:, :w]
                    ibase = C.cast(r.iq_out, C.c_void_p).value
                    iqo = np.frombuffer(device_to_host(ibase, 8 * c * stride), np.float32).reshape(c, stride, 2)[:, :w]
                else:
                    wave = np.ctypeslib.as_array(r.waveout, shape=(c, stride))[:, :w]
                    iqo = np.ctypeslib.as_array(r.iq_out, shape=(c, stride, 2))[:, :w]
                st = np.ctypeslib.as_array(C.cast(r.status, C.POINTER(C.c_uint32)), shape=(nb, c, 10))
                for a in (wave, iqo, st):
                    h.update(np.ascontiguousarray(a).tobytes())
                digests.append((nb, r.frames_done, h.hexdigest()))
    finally:
        e.close()
    return digests


@pytest.mark.gpu
def test_cfg4_full_size_split_over_two_members(cuda):
    """Full-size cfg 4 for 2 signal-seconds with its channels alternately on two members of GPU 0: audio, status and
    iq_out equal one engine's, bit for bit, with results in pinned host memory and left on the device."""
    alt = [c % 2 for c in range(2000)]
    want = run_cfg4(cuda, 2.0)
    assert sum(nb for nb, _, _ in want) >= 15
    assert run_cfg4(cuda, 2.0, [0, 0], alt) == want
    on_dev = run_cfg4(cuda, 2.0, [0, 0], alt, flags=abi.FLAG_RESULTS_ON_DEVICE)
    assert on_dev == run_cfg4(cuda, 2.0, flags=abi.FLAG_RESULTS_ON_DEVICE) == want


@pytest.mark.gpu
def test_split_over_two_gpus(cuda):
    """The main scenario and full-size cfg 4 over GPUs 0 and 1 (NVLink peer stores), where two GPUs are visible."""
    if visible_gpus() < 2:
        pytest.skip("one GPU visible: the split over two GPUs (peer stores between GPUs) needs at least two")
    from boondock_airband_b200.engine import Engine
    cfg, streams = scenario(0.9)
    one = Engine(cfg, cuda)
    want = drive(one, cfg, streams, (1_300_007, 500_003, 400_001), 3)
    one.close()
    g = Engine(cfg, cuda, gpus=[0, 1, 0], gpu_of_device=GPU_OF_DEVICE, gpu_of_channel=split_map(cfg))
    got = drive(g, cfg, streams, (1_300_007, 500_003, 400_001), 3)
    g.close()
    assert_same(got, want, cfg)
    assert run_cfg4(cuda, 2.0, [0, 1], [c % 2 for c in range(2000)]) == run_cfg4(cuda, 2.0)
