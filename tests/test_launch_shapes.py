"""The launch shapes the workloads run, compared with plain references, on the thread-emulated build ("emu", CPU) and on a
B200 ("cuda", -m gpu).

A. The channelizer's streaming path (K1: persistent CTAs, tiles off a launch-wide counter, the next tile's bytes prefetched
   into the other half of a double buffer, pick table reloaded when a CTA moves to another input) at every FFT size and
   sample format, with enough inputs that every resident CTA takes several tiles per step: picked bins against a float64
   DFT, replicas against their source bit for bit, other tilings bit for bit, K1's magnitudes through the demodulator.
B. The demodulator's many-channel launch shapes (demod_full_kernel<4>, the plain kernel spread over several lanes per CTA
   with a partial last CTA, the plain kernel packed beside the general one) fed the oracle's picks: bit-exact.

Every scenario is sized from the SM count the library sees (the emulation reports 2), and every test asserts that the
shape it is named for was reached, through restatements of the engine's launch rules below."""
import copy

import numpy as np
import pytest

from boondock_airband_b200 import abi, synth
from boondock_airband_b200.abi import ChannelCfg, DeviceCfg, EngineCfg
from boondock_airband_b200.engine import Engine
from oracle.ba_oracle import Oracle

import parity
import scenarios

LIBS = ["emu", pytest.param("cuda", marks=pytest.mark.gpu)]

EMU_SMS = 2                  # tests/emu/cuda_emu.h: cudaDevAttrMultiProcessorCount
EMU_SMEM_OPTIN = 227 * 1024  # ... and cudaDevAttrMaxSharedMemoryPerBlockOptin


@pytest.fixture(scope="module")
def libs(oracle_built):
    return {}


def library(libs, kind):
    """(library path, SM count, opt-in shared memory per block) of the library `kind` runs on."""
    if kind not in libs:
        if kind == "emu":
            libs[kind] = (parity.lib_for("emu"), EMU_SMS, EMU_SMEM_OPTIN)
        else:
            import torch
            prop = torch.cuda.get_device_properties(0)
            libs[kind] = (parity.lib_for("cuda"), prop.multi_processor_count, prop.shared_memory_per_block_optin)
    return libs[kind]


# ---------------------------------------------------------------------------------------------------------------- launch rules

# channelize.cu:58-63, BA_PLAN: values per thread, threads per CTA, resident CTAs per SM the register cap is chosen for
K1_PLAN = {256: (16, 256, 2), 512: (32, 128, 3), 1024: (32, 128, 2), 2048: (16, 256, 2), 4096: (16, 256, 2), 8192: (32, 256, 2)}


def k1_groups(n):
    v, threads, _ = K1_PLAN[n]
    return threads // (n // v)


def k1_smem_bytes(n, raw_bytes, max_channels):
    """channelize.cu:784-786."""
    return 2 * raw_bytes + 8 * k1_groups(n) * (n + n // 8) + 2 * ((max_channels + 7) & ~7) + 64


def sample_bytes(dev):
    return 2 * dev.bytes_per_sample


def hop_bytes(cfg, dev):
    """ba_engine.cu:648: bytes per complex sample times round(sample_rate / wave_rate)."""
    return sample_bytes(dev) * int(round(dev.sample_rate / cfg.wave_rate))


def k1_tiling(cfg, sms, smem_optin, tile_env=None, ctas_env=None):
    """(frames per tile, resident K1 CTAs) the engine picks: restates choose_tiles (ba_engine.cu:473-517) and the grid of
    the launch (ba_engine.cu:1410, min(tiles, SMs x CTAs per SM))."""
    n = cfg.fft_size
    groups = k1_groups(n)
    ctas = K1_PLAN[n][2] if ctas_env is None else max(1, ctas_env)
    max_hop = max(hop_bytes(cfg, d) for d in cfg.devices)
    max_frame = max(sample_bytes(d) * n for d in cfg.devices)
    fixed = k1_smem_bytes(n, 0, max(len(d.channels) for d in cfg.devices))
    budget = min(smem_optin, 216 * 1024 // ctas if ctas > 2 else 96 * 1024)

    def raw_of(tf):
        return ((tf - 1) * max_hop + max_frame + 32 + 15) & ~15

    tf = 4 * groups
    frames_per_step = len(cfg.devices) * cfg.max_batches_per_step * (cfg.wave_rate // 8)
    if frames_per_step // (6 * groups) >= 16 * sms * ctas:
        tf = 6 * groups
    if tile_env is not None:
        tf = max(groups, tile_env // groups * groups)
    if n == 8192:  # k1_direct: frames straight from global memory
        return (tf if tile_env is not None else 4), sms * ctas
    while tf > groups and fixed + 2 * raw_of(tf) > budget:
        tf -= groups
    while tf > 1 and fixed + 2 * raw_of(tf) > smem_optin:
        tf -= 1
    if tf > 1:
        tf &= ~1
    assert fixed + 2 * raw_of(tf) <= smem_optin
    return tf, sms * ctas


def is_plain(cfg, ch):
    """ba_engine.cu:753-759: channels of demod_plain_kernel (AM without options, no trace)."""
    return (ch.modulation == "am" and not ch.bandwidth and not ch.notch and not ch.ctcss and not ch.has_iq_outputs and not ch.afc
            and not ch.freqs and not (cfg.flags & abi.FLAG_TRACE))


def k2_shape(cfg, sms):
    """What k2_launch (demod.cu:2407-2452) launches for this engine: the general kernel's build and the plain kernel's channels
    per CTA (`lanes`), CTAs, and whether it runs beside the general kernel (second stream)."""
    chans = [c for d in cfg.devices for c in d.channels]
    n_plain = sum(is_plain(cfg, c) for c in chans)
    n_full = len(chans) - n_plain
    shape = dict(n_plain=n_plain, n_full=n_full, full=None, lanes=0, plain_ctas=0, beside=n_plain > 0 and n_full > 0)
    if n_full:
        shape["full"] = 4 if n_full > 3 * sms else 1
    if n_plain:
        lanes = 32 if n_full else min(32, max(1, -(-n_plain // (2 * sms))))
        shape["lanes"] = lanes
        shape["plain_ctas"] = -(-n_plain // lanes)
    return shape


# ---------------------------------------------------------------------------------------------------------------- A. channelizer

# (format, sample rate, centre): four sources with distinct rates, each an exact multiple of the 8 kHz wave rate
K1_SOURCES = (("u8", 2_560_000, 120_000_000), ("s8", 2_048_000, 131_000_000), ("s16", 2_400_000, 145_000_000), ("f32", 1_920_000, 460_000_000))
K1_SECONDS = 0.3
K1_FIRST = 151        # frames of the first step (odd: every later launch starts on an odd frame of the stream)
K1_CHUNK = 1100       # frames per submitted piece after the first (plus a ragged 7 bytes)
K1_TILES_PER_CTA = 4


def k1_source_devices():
    """Receivers of 16 AM channels per source (plain ones, one through the low-pass, one with iq_out, one at a manual
    squelch level), and the transmitters that put carriers on 11 of them: 5 channels listen to noise."""
    rx, tx = [], []
    for i, (fmt, fs, cf) in enumerate(K1_SOURCES):
        freqs = [cf + int((k - 7.5) * 110_000) + 3_000 * i for k in range(16)]
        ch = [ChannelCfg(freq=f) for f in freqs]
        ch[3].bandwidth = 6000
        ch[8].has_iq_outputs = True
        ch[12].squelch_threshold = -40
        # s16 at a full scale of 2^15 so that x / 32768 is the exact conversion (the default 32766.5 is not a power of two)
        fullscale = 32768.0 if fmt == "s16" else None
        rx.append(DeviceCfg(sample_rate=fs, centerfreq=cf, sample_format=fmt, fullscale=fullscale, channels=ch))
        tx.append(DeviceCfg(sample_rate=fs, centerfreq=cf, sample_format=fmt, channels=[ChannelCfg(freq=f) for k, f in enumerate(freqs) if k % 3 != 2]))
    return rx, tx


_K1_STREAMS = {}


def k1_streams():
    if not _K1_STREAMS:
        _, tx = k1_source_devices()
        for i, d in enumerate(tx):
            _K1_STREAMS[i] = synth.synth(d, K1_SECONDS, 60 + i, gate_on=0.12, gate_off=0.05)
    return [_K1_STREAMS[i] for i in range(len(K1_SOURCES))]


def k1_config(n, replicas):
    rx, _ = k1_source_devices()
    return EngineCfg(fft_size=n, wave_rate=8000, devices=[copy.deepcopy(rx[i % len(rx)]) for i in range(replicas * len(rx))],
                     flags=abi.FLAG_KEEP_PICKS, max_batches_per_step=2)


def k1_replicas(n, sms, smem_optin):
    """Fewest copies of the four sources that give one step of K1_CHUNK frames per input K1_TILES_PER_CTA tiles per resident
    CTA."""
    for r in range(1, 64):
        tf, resident = k1_tiling(k1_config(n, r), sms, smem_optin)
        if r * len(K1_SOURCES) * -(-K1_CHUNK // tf) >= K1_TILES_PER_CTA * resident:
            return r
    raise AssertionError("no replica count reaches %d tiles per CTA" % K1_TILES_PER_CTA)


def stream_with_picks(cfg, streams, lib, shift=0):
    """Feed the inputs (first step: K1_FIRST frames, plus one on every other copy of the sources and plus `shift`; then ragged
    pieces of about K1_CHUNK frames) and read every input's picked bins after every step, while they are in the ring.  Copies
    of one source thus start their later launches on frames of either parity.  Returns (results as run_stream, picks [input] -> [C][frames] complex64,
    frames per input of every step)."""
    e = Engine(cfg, lib)
    try:
        nd = len(cfg.devices)
        views = [np.ascontiguousarray(streams[d % len(streams)]).view(np.uint8).reshape(-1) for d in range(nd)]
        firsts = [K1_FIRST + shift + (d // len(streams)) % 2 for d in range(nd)]
        hops = [hop_bytes(cfg, d) for d in cfg.devices]
        picks = [[[] for _ in d.channels] for d in cfg.devices]
        steps = []
        acc = e._new_acc()
        first = True
        pos = [0] * nd
        while True:
            fed = False
            for d in range(nd):
                want = firsts[d] * hops[d] + sample_bytes(cfg.devices[d]) * cfg.fft_size if first else K1_CHUNK * hops[d] + 7
                k = min(want, views[d].size - pos[d], e.input_space(d))
                if k > 0:
                    e.submit(d, views[d][pos[d]:pos[d] + k])
                    pos[d] += k
                    fed = True
            before = [a["frames_done"] for a in acc]
            produced, advanced = e._step_into(acc)
            now = [a["frames_done"] for a in acc]
            if first:
                assert now == firsts, (now, firsts)
                first = False
            steps.append([b - a for a, b in zip(before, now)])
            for d in range(nd):
                if now[d] > before[d]:
                    for c in range(len(cfg.devices[d].channels)):
                        p = e.debug_picks(d, c, before[d], now[d] - before[d])
                        picks[d][c].append(p[:, 0] + 1j * p[:, 1])
            if not fed and not produced and not advanced:
                break
        res = e._finish_acc(acc)
    finally:
        e.close()
    picks = [np.stack([np.concatenate(pc) for pc in pd]).astype(np.complex64) for pd in picks]
    return res, picks, steps


def exact_samples(dev, iq):
    """Interleaved raw samples -> complex128, converted exactly: u8 (x - 127.5) / 127.5, s8 x / 128, s16 x / full scale, f32 as is."""
    x = iq.astype(np.float64)
    if dev.sample_format == "u8":
        x = (x - 127.5) / 127.5
    elif dev.sample_format == "s8":
        x = x / 128.0
    elif dev.sample_format == "s16":
        x = x / dev.default_fullscale()
    return x[0::2] + 1j * x[1::2]


def dft_at_bins(dev, iq, n, hop, window, bins, frames, first=0, chunk=256):
    """float64 DFT of frames [first, first + frames) at `bins` only: [frames][len(bins)] plus each windowed frame's L2 norm
    (= the RMS of its spectrum)."""
    z = exact_samples(dev, iq)
    w = window.astype(np.float64)
    kern = np.exp(-2j * np.pi * np.outer(np.arange(n), np.asarray(bins)) / n)
    out = np.empty((frames, len(bins)), np.complex128)
    norm = np.empty(frames)
    for f0 in range(0, frames, chunk):
        f1 = min(frames, f0 + chunk)
        idx = (first + np.arange(f0, f1))[:, None] * hop + np.arange(n)[None, :]
        x = z[idx] * w
        out[f0:f1] = x @ kern
        norm[f0:f1] = np.sqrt((np.abs(x) ** 2).sum(axis=1))
    return out, norm


def oracle_fft_level(cfg, dev, iq, window, n_frames=24):
    """The float32 FFT of the CPU oracle against the float64 DFT on `n_frames` frames from the middle of the stream: the
    largest error at any bin over the frame's L2 norm."""
    n = cfg.fft_size
    hop = hop_bytes(cfg, dev) // sample_bytes(dev)
    one = copy.copy(cfg)
    one.devices = [dev]
    first = (len(iq) // 2 // hop) // 2
    part = iq[2 * first * hop:2 * (first * hop + (n_frames - 1) * hop + n)]
    o = Oracle(one)
    try:
        _, fo = o.debug_frames(0, part, n_frames, want_in=False)
    finally:
        o.close()
    z = exact_samples(dev, iq)
    x = z[(first + np.arange(n_frames))[:, None] * hop + np.arange(n)[None, :]] * window.astype(np.float64)
    ref, norm = np.fft.fft(x, axis=1), np.sqrt((np.abs(x) ** 2).sum(axis=1))
    got = fo[..., 0].astype(np.float64) + 1j * fo[..., 1]
    return float((np.abs(got - ref) / norm[:, None]).max())


def check_inject_equals_stream(cfg, picks, streamed, lib, frames_per_call=1777):
    """A second engine fed the streamed engine's own picks (magnitudes computed on the host with IEEE operations) must
    deliver the same audio, iq_out and status bit for bit: K1's magnitudes equal |pick| as the demodulator needs them."""
    e = Engine(cfg, lib)
    try:
        nd = len(cfg.devices)
        stacked = [np.stack([p.real, p.imag], axis=-1).transpose(1, 0, 2).astype(np.float32) for p in picks]  # [frames][C][2]
        pos = [0] * nd
        acc = e._new_acc()
        while True:
            fed = False
            for d in range(nd):
                if pos[d] < stacked[d].shape[0]:
                    k = min(frames_per_call, stacked[d].shape[0] - pos[d])
                    e.inject_picks(d, stacked[d][pos[d]:pos[d] + k])
                    pos[d] += k
                    fed = True
            produced, advanced = e._step_into(acc)
            if not fed and not produced and not advanced:
                break
        got = e._finish_acc(acc)
    finally:
        e.close()
    for d in range(len(cfg.devices)):
        assert_same_results(streamed[d], got[d], "input %d, injected vs streamed" % d)


def assert_same_results(a, b, what):
    assert a["frames_done"] == b["frames_done"], (what, a["frames_done"], b["frames_done"])
    assert np.array_equal(a["waveout"].view(np.uint32), b["waveout"].view(np.uint32)), what + ": audio differs"
    for key in ("iq_out", "trace"):
        assert (a[key] is None) == (b[key] is None), (what, key)
        if a[key] is not None:
            assert np.array_equal(a[key].view(np.uint8), b[key].view(np.uint8)), "%s: %s differs" % (what, key)
    assert a["status"] == b["status"], what + ": status rows differ"


PICK_ERRORS = {}  # (kind, n, format) -> (peak-relative, over the frame norm, oracle's level): printed by -s runs


@pytest.mark.parametrize("kind", LIBS)
@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192])
def test_channelizer_streaming_every_size_and_format(libs, kind, n, monkeypatch):
    lib, sms, optin = library(libs, kind)
    for var in ("BA_CUDA_K1_TILE", "BA_CUDA_K1_CTAS", "BA_CUDA_SERIAL_K2"):
        monkeypatch.delenv(var, raising=False)
    streams = k1_streams()
    ns = len(streams)
    r = k1_replicas(n, sms, optin)
    cfg = k1_config(n, r)
    tf, resident = k1_tiling(cfg, sms, optin)
    res, picks, steps = stream_with_picks(cfg, streams, lib)

    # the shape: some step gave every resident CTA K1_TILES_PER_CTA tiles or more
    tiles = max(sum(-(-f // tf) for f in step) for step in steps)
    assert tiles >= K1_TILES_PER_CTA * resident, (tiles, tf, resident, steps)

    # every replica computes what its source computes, bit for bit (its tiles land on other CTAs and buffer halves)
    for d in range(ns, len(cfg.devices)):
        assert np.array_equal(picks[d].view(np.uint32), picks[d % ns].view(np.uint32)), "input %d: picks differ from its source" % d
        assert_same_results(res[d % ns], res[d], "input %d, replica vs source" % d)

    # picked bins against the float64 DFT of the exactly converted samples
    e = Engine(cfg, lib)
    window = e.window()
    bins = [[e.channel_info(s, c).bin for c in range(len(cfg.devices[s].channels))] for s in range(ns)]
    e.close()
    for s in range(ns):
        dev = cfg.devices[s]
        frames = res[s]["frames_done"]
        assert picks[s].shape == (len(dev.channels), frames)
        hop = hop_bytes(cfg, dev) // sample_bytes(dev)
        ref, norm = dft_at_bins(dev, streams[s], n, hop, window, bins[s], frames)
        err = np.abs(picks[s].T.astype(np.complex128) - ref)
        peak = float((err / np.abs(ref).max(axis=0)).max())
        rms = float((err / norm[:, None]).max())
        level = oracle_fft_level(cfg, dev, streams[s], window)
        PICK_ERRORS[(kind, n, dev.sample_format)] = (peak, rms, level)
        assert peak <= parity.TOL_BASEBAND, (dev.sample_format, peak)
        assert rms <= 8 * level, (dev.sample_format, rms, level)

    # other tilings (one round of FFT groups per tile, one CTA per SM), the first with a first step one frame longer: the
    # same picks and audio bit for bit
    for var, value, shift in (("BA_CUDA_K1_TILE", 1, 1), ("BA_CUDA_K1_CTAS", 1, 0)):
        monkeypatch.setenv(var, str(value))
        other, other_picks, _ = stream_with_picks(cfg, streams, lib, shift)
        monkeypatch.delenv(var)
        for d in range(len(cfg.devices)):
            assert np.array_equal(other_picks[d].view(np.uint32), picks[d].view(np.uint32)), "%s=%d: input %d picks differ" % (var, value, d)
            assert_same_results(res[d], other[d], "%s=%d: input %d" % (var, value, d))

    # K1's magnitudes: the demodulator fed the same picks through the host gives the same results
    check_inject_equals_stream(cfg, picks, res, lib)

    # one input per source end to end against the oracle, at the stated bars
    one = copy.copy(cfg)
    one.devices = cfg.devices[:ns]
    one.flags = abi.FLAG_TRACE
    o = Oracle(one)
    try:
        for s in range(ns):
            o.feed(s, streams[s])
        parity.compare_streams(one, o, res[:ns], min_open=500)
    finally:
        o.close()
    print("\nN=%d tiles of %d frames, %d inputs, %d resident CTAs, %d tiles in the largest step; pick errors: %s" % (
        n, tf, len(cfg.devices), resident, tiles,
        ", ".join("%s %.2e/%.2e (oracle %.2e)" % (f, *PICK_ERRORS[(kind, n, f)]) for f, _, _ in K1_SOURCES)))


# ---------------------------------------------------------------------------------------------------------------- B. demodulator

def check_demod_exact_replicas(cfg, sources, layout, lib, frames_per_call=(1777,)):
    """check_demod_exact for engines whose inputs are copies of a few sources: the oracle runs once per source
    (sources[i] = (DeviceCfg, stream)); engine input d is a copy of source layout[d] and is fed that source's picks,
    frames_per_call[d % len(frames_per_call)] frames per call.  Every input's audio, trace, iq_out, levels and counters
    must equal its source's oracle output bit for bit."""
    oracles, picks = [], []
    for dev, stream in sources:
        one = copy.copy(cfg)
        one.devices = [dev]
        one.flags = cfg.flags | abi.FLAG_TRACE  # the oracle records picks and decisions only when asked to trace
        o = Oracle(one)
        o.feed(0, stream)
        oracles.append((one, o))
        picks.append(np.stack([o.picks(0, c) for c in range(len(dev.channels))], axis=1))  # [frames][C][2]
    e = Engine(cfg, lib)
    try:
        nd = len(cfg.devices)
        pos = [0] * nd
        acc = e._new_acc()
        while True:
            fed = False
            for d in range(nd):
                p = picks[layout[d]]
                if pos[d] < p.shape[0]:
                    k = min(frames_per_call[d % len(frames_per_call)], p.shape[0] - pos[d])
                    e.inject_picks(d, p[pos[d]:pos[d] + k])
                    pos[d] += k
                    fed = True
            produced, advanced = e._step_into(acc)
            if not fed and not produced and not advanced:
                break
        res = e._finish_acc(acc)
    finally:
        e.close()
    try:
        for d in range(nd):
            one, o = oracles[layout[d]]
            parity.compare_streams(one, o, [res[d]], exact=True)
    finally:
        for _, o in oracles:
            o.close()
    return res


def plain_stress_sources(seconds):
    """Three inputs of different formats, rates and lengths with 7, 6 and 4 plain AM channels driven as scenarios.am_stress
    does: carriers from strong to below the squelch threshold, an amplitude step in every transmission, 130 ms transmissions
    40 ms apart - lanes of one warp take different squelch paths in the same chunk."""
    levels = [-25.0, -35.0, -44.0, -46.0, -47.0, -48.0, -49.0, -50.0]
    out = []
    for i, (fmt, fs, cf, nch, length) in enumerate((("u8", 2_560_000, 120_000_000, 7, 1.0), ("s8", 2_048_000, 131_000_000, 6, 0.75),
                                                    ("s16", 2_400_000, 145_000_000, 4, 0.55))):
        dev = DeviceCfg(sample_rate=fs, centerfreq=cf, sample_format=fmt, channels=[ChannelCfg(freq=cf + (k - 3) * 140_000 + 7_000 * i) for k in range(nch)])
        iq = synth.synth(dev, seconds * length, 80 + i, gate_on=0.13, gate_off=0.04, am_depth=0.9, carrier_dbfs=levels[i:i + nch], burst=3.0)
        out.append((dev, iq))
    return out


def replicate(sources, counts, **kw):
    """Engine configuration whose inputs are counts[i] copies of sources[i]; returns (cfg, layout)."""
    layout = [i for i, n in enumerate(counts) for _ in range(n)]
    cfg = EngineCfg(fft_size=512, wave_rate=8000, devices=[copy.deepcopy(sources[i][0]) for i in layout], **kw)
    return cfg, layout


@pytest.mark.parametrize("kind", LIBS)
@pytest.mark.parametrize("fm_demod", [abi.FM_FAST_ATAN2, abi.FM_QUADRI_DEMOD])
def test_general_kernel_four_ctas_per_sm_exact(libs, kind, fm_demod):
    """More general channels than three CTAs per SM hold: demod_full_kernel<4> on every option of scenarios.mixed_options
    but AFC (NFM with and without the low-pass, CTCSS with notch, AM through the low-pass, iq_out, manual squelch)."""
    lib, sms, _ = library(libs, kind)
    cfg0, streams = scenarios.mixed_options(0.45, fm_demod=fm_demod, afc=False)
    per = len(cfg0.devices[0].channels)
    copies = max(2, -(-(3 * sms + 1) // per))
    cfg = copy.copy(cfg0)
    cfg.devices = [copy.deepcopy(cfg0.devices[0]) for _ in range(copies)]
    shape = k2_shape(cfg, sms)
    assert shape["n_plain"] == 0 and shape["full"] == 4 and shape["n_full"] > 3 * sms, shape
    check_demod_exact_replicas(cfg, [(cfg0.devices[0], streams[0])], [0] * copies, lib, frames_per_call=(1777, 1213, 2001))


def plain_spread_config(sms, seconds):
    sources = plain_stress_sources(seconds)
    per = sum(len(d.channels) for d, _ in sources)
    for r in range(2, 200):  # more than 6 x SMs plain channels whose count leaves the last CTA of the spread launch partial
        cfg, layout = replicate(sources, [r] * len(sources), max_batches_per_step=3)
        shape = k2_shape(cfg, sms)
        if r * per > 6 * sms and shape["n_plain"] % shape["lanes"]:
            return sources, cfg, layout, shape
    raise AssertionError("no replica count gives a partial last CTA")


@pytest.mark.parametrize("kind", LIBS)
def test_plain_kernel_spread_lanes_exact(libs, kind, monkeypatch):
    """Plain channels only, spread over the SMs with several channels per CTA and a partial last CTA; the inputs differ in
    rate and length and are fed unevenly, so lanes of one CTA deliver different batch counts, some none, in a step.  The
    result does not depend on whether the demodulator runs beside or behind the channelizer (BA_CUDA_SERIAL_K2)."""
    lib, sms, _ = library(libs, kind)
    sources, cfg, layout, shape = plain_spread_config(sms, 1.0)
    assert shape["n_full"] == 0 and 1 < shape["lanes"] < 32 and shape["n_plain"] > 2 * sms, shape
    assert shape["n_plain"] % shape["lanes"] != 0, shape
    runs = []
    for serial in ("0", "1"):
        monkeypatch.setenv("BA_CUDA_SERIAL_K2", serial)
        runs.append(check_demod_exact_replicas(cfg, sources, layout, lib, frames_per_call=(1777, 1001, 2333, 1499)))
    monkeypatch.delenv("BA_CUDA_SERIAL_K2")
    for d in range(len(cfg.devices)):
        assert_same_results(runs[0][d], runs[1][d], "input %d, BA_CUDA_SERIAL_K2=0 vs 1" % d)
        assert float(np.abs(runs[0][d]["waveout"]).max()) > 0.05


@pytest.mark.parametrize("kind", LIBS)
def test_plain_kernel_packed_beside_general_exact(libs, kind):
    """Plain AM channels in two full warps and a partial one (demod_plain_kernel packed 32 to a CTA, on the second stream)
    next to a few general channels (demod_full_kernel, first stream)."""
    lib, sms, _ = library(libs, kind)
    sources = plain_stress_sources(0.8)
    cf = 460_000_000
    general = DeviceCfg(sample_rate=1_920_000, centerfreq=cf, sample_format="f32", channels=[
        ChannelCfg(freq=cf - 300_000, bandwidth=6000), ChannelCfg(freq=cf - 100_000, notch=1000.0, notch_q=5.0),
        ChannelCfg(freq=cf + 200_000, has_iq_outputs=True), ChannelCfg(freq=cf + 400_000)])
    sources.append((general, synth.synth(general, 0.7, 90, gate_on=0.2, gate_off=0.07)))
    cfg, layout = replicate(sources, [4, 4, 4, 1], max_batches_per_step=3)
    shape = k2_shape(cfg, sms)
    assert shape["beside"] and shape["lanes"] == 32 and 64 < shape["n_plain"] < 96 and 0 < shape["n_full"] <= 3 * sms, shape
    check_demod_exact_replicas(cfg, sources, layout, lib, frames_per_call=(1777, 1001, 2333))
