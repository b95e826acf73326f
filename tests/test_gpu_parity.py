"""Parity of the CUDA path (libba_cuda.so through its C-ABI) with the CPU oracle, on a B200.

Bars (BASELINE.json north_star): sample conversion, bin indices and squelch decisions bit-exact; channel baseband
(picked-bin IQ) within 1e-4 relative; demodulated audio within 1e-3.  Given identical picked-bin IQ the demodulator is
required to be bit-exact in everything (audio, iq_out, levels, counters)."""
import numpy as np
import pytest

from boondock_airband_b200 import abi, configs, synth
from boondock_airband_b200.abi import ChannelCfg, DeviceCfg, EngineCfg
from boondock_airband_b200.engine import Engine, EngineError

import parity
import scenarios

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cuda(oracle_built):
    return parity.lib_for("cuda")


@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192])
@pytest.mark.parametrize("fmt", ["u8", "s8", "s16", "f32"])
def test_frames(cuda, n, fmt):
    rng = np.random.default_rng(n + len(fmt))
    dev = DeviceCfg(sample_rate=2_400_000, centerfreq=100_000_000, sample_format=fmt,
                    channels=[ChannelCfg(freq=100_000_000 + 12_500 * k) for k in range(-5, 6)])
    cfg = EngineCfg(fft_size=n, wave_rate=16000, devices=[dev])
    nfr = 70
    iq = parity.random_iq(rng, fmt, 150 * (nfr - 1) + n + 5)
    parity.check_frames(cfg, iq, nfr, cuda)


def test_u8_all_codes(cuda):
    dev = DeviceCfg(sample_rate=2_560_000, centerfreq=120_000_000, channels=[ChannelCfg(freq=120_100_000)])
    cfg = EngineCfg(fft_size=256, wave_rate=8000, devices=[dev])
    base = np.repeat(np.arange(256, dtype=np.uint8), 2)
    iq = np.resize(np.concatenate([base, base[::-1]]), 2 * (320 * 7 + 256)).astype(np.uint8)
    parity.check_frames(cfg, iq, 8, cuda)


@pytest.mark.parametrize("which", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_channel_constants(cuda, which):
    """Bin indices (config.cpp:669-670), dm_dphi (:682-715) and filter/squelch/CTCSS constants, all workloads."""
    cfg = {"cfg1": configs.cfg1, "cfg2": configs.cfg2, "cfg3": lambda: configs.cfg3(4), "cfg4": lambda: configs.cfg4(400),
           "cfg5": lambda: configs.cfg5(4, 2048)}[which]()
    parity.check_channel_info(cfg, cuda)


def test_cfg1(cuda):
    cfg, streams = scenarios.cfg1_short(2.1)
    o, res, launches = parity.run_both(cfg, streams, cuda, chunk_bytes=700_001)
    parity.compare_streams(cfg, o, res, min_open=5000)
    assert launches > 0


def test_cfg1_fast_path(cuda):
    """Without the trace flag plain AM channels take the specialised (PLAIN) instantiation of the demodulator."""
    cfg, streams = scenarios.cfg1_short(2.1)
    cfg.flags = 0
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=700_001)
    assert res[0]["trace"] is None
    parity.compare_streams(cfg, o, res)
    assert float(np.abs(res[0]["waveout"]).max()) > 0.05


def test_fast_path_bit_exact(cuda):
    """The PLAIN instantiation fed with the oracle's picks: audio and levels bit-exact (trace is compared through the audio gate)."""
    cfg, streams = scenarios.cfg1_short(1.2)
    from oracle.ba_oracle import Oracle
    o = Oracle(cfg)
    o.feed(0, streams[0])
    picks = np.stack([o.picks(0, c) for c in range(8)], axis=1)
    cfg.flags = 0
    e = Engine(cfg, cuda)
    waves = []
    for lo in range(0, picks.shape[0], 2500):
        e.inject_picks(0, picks[lo:lo + 2500])
        t = e.process()
        r = e.collect(t, 0)
        if r.n_batches:
            waves.append(r.waveout)
    e.close()
    got = np.concatenate(waves, axis=1)
    for c in range(8):
        assert np.array_equal(got[c].view(np.uint32), o.waveout(0, c).view(np.uint32)), c


def test_plain_kernel_exact(cuda):
    """demod_plain_kernel fed with the oracle's picks: audio, levels and counters bit-exact (ragged frame counts per call)."""
    cfg, streams = scenarios.cfg1_short(2.1)
    cfg.flags = 0
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=2777)


@pytest.mark.parametrize("frames_per_call", [1100, 2777, 8000])
def test_plain_kernel_stress_exact(cuda, frames_per_call):
    """The speculative quad path of demod_plain_kernel against the sequential loop on marginal, flapping, clipping
    carriers (every squelch state, flap detection, low-signal aborts, AGC clip): bit-exact."""
    cfg, streams = scenarios.am_stress(3.0)
    cfg.flags = 0
    cfg.max_batches_per_step = 8
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=frames_per_call)


def test_general_kernel_stress_exact(cuda):
    """Same stimulus through the general kernel (trace on)."""
    cfg, streams = scenarios.am_stress(2.0)
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=2777)


def test_cfg1_picks(cuda):
    cfg, streams = scenarios.cfg1_short(0.4)
    parity.check_picks(cfg, streams[0][:2_000_000], cuda)


def test_cfg2(cuda):
    cfg, streams = scenarios.cfg2_small(32, 2.0)
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=2_000_003)
    parity.compare_streams(cfg, o, res, min_open=5000)
    # CTCSS windows completed and both outcomes occurred
    hits = sum(res[0]["status"][-1][c]["ctcss_count"] for c in range(32))
    misses = sum(res[0]["status"][-1][c]["no_ctcss_count"] for c in range(32))
    assert hits > 0 and misses > 0


def test_cfg2_picks(cuda):
    cfg, streams = scenarios.cfg2_small(32, 0.3)
    parity.check_picks(cfg, streams[0][:1_200_000], cuda)


@pytest.mark.parametrize("fm_demod", [abi.FM_FAST_ATAN2, abi.FM_QUADRI_DEMOD])
def test_demod_bit_exact(cuda, fm_demod):
    cfg, streams = scenarios.mixed_options(1.5, fm_demod=fm_demod, afc=False)
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=3777)


@pytest.mark.parametrize("fm_demod", [abi.FM_FAST_ATAN2, abi.FM_QUADRI_DEMOD])
def test_demod_bit_exact_squelch_held_by_the_filtered_average(cuda, fm_demod):
    """The chunk-at-a-time paths for a squelch that only counts (held CLOSED with every sample filtered, OPENING, LOW_SIGNAL_ABORT)
    against the oracle's sequential loop, bit for bit; the oracle's trace is required to show thousands of samples in each."""
    cfg, streams = scenarios.held_by_post_filter(1.6, fm_demod=fm_demod)
    parity.require_squelch_regimes(cfg, streams)
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=3333)
    cfg.flags = 0  # and without the trace (the stores of the silent kinds differ)
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=2000)


def test_demod_bit_exact_cfg2(cuda):
    cfg, streams = scenarios.cfg2_small(16, 1.6)
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=3000)


def test_mixed_options_end_to_end(cuda):
    cfg, streams = scenarios.mixed_options(1.5)
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=555_555)
    parity.compare_streams(cfg, o, res, min_open=3000)


def check_afc_walk(cfg, o, res):
    """Every branch of AFC::finalize (.cpp:222-250) ran, on the engine exactly as on the oracle (compare_streams has already
    required equal bin and axcindicate for every batch): an upward walk, a downward walk, and the restore of base_bins on
    the open -> closed edge, more than once."""
    rows = res[0]["status"]
    base = [o.channel_info(0, c).bin for c in range(len(cfg.devices[0].channels))]
    seen = {c: [(r[c]["axcindicate"], r[c]["bin"]) for r in rows] for c in range(len(base))}
    assert any(a == abi.AFC_UP and b > base[0] for a, b in seen[0]), seen[0]
    assert any(a == abi.AFC_DOWN and b < base[1] for a, b in seen[1]), seen[1]
    assert all(b == base[4] for _, b in seen[4])  # the walk finds no stronger neighbour: never moves
    restores = walks = 0
    for c in range(len(base)):
        moved = [b != base[c] for _, b in seen[c]]
        walks += sum(1 for k in range(1, len(moved)) if not moved[k - 1] and moved[k]) + (1 if moved[0] else 0)
        for k in range(1, len(moved)):
            if moved[k - 1] and not moved[k]:
                restores += 1
                assert seen[c][k][0] == abi.NO_SIGNAL  # the restore happens on the batch in which the channel went silent
    assert restores >= 4 and walks >= 7, (restores, walks, seen)


def test_afc_walks_up_down_and_restores(cuda):
    cfg, streams = scenarios.afc_walk(1.7)
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=777_777)
    parity.compare_streams(cfg, o, res, min_open=3000)
    check_afc_walk(cfg, o, res)


def test_s8_code_0x80(cuda):
    """levels_s8[(uint8_t)i] = i / 128.0f is filled for i in -127..127 only (boondock_airband.cpp:344-346): the entry of byte
    0x80 is whatever the stack held.  Engine and oracle both define it as -128 / 128 = -1.0 (the value the formula gives
    when continued); a frame made of every byte value, 0x80 included, converts bit-exactly."""
    dev = DeviceCfg(sample_rate=2_560_000, centerfreq=120_000_000, sample_format="s8", channels=[ChannelCfg(freq=120_100_000)])
    cfg = EngineCfg(fft_size=256, wave_rate=8000, devices=[dev])
    base = np.repeat(np.arange(-128, 128, dtype=np.int16).astype(np.int8), 2)
    iq = np.resize(np.concatenate([base, base[::-1]]), 2 * (320 * 7 + 256)).astype(np.int8)
    assert (iq == -128).any()
    parity.check_frames(cfg, iq, 8, cuda)
    e = Engine(cfg, cuda)
    fi, _ = e.debug_frames(0, iq, 1)
    e.close()
    w = e.window() if False else None
    k = int(np.where(iq[:512:2] == -128)[0][0])
    from oracle.ba_oracle import Oracle
    win = Oracle(cfg).window()
    assert fi[0, k, 0] == np.float32(-1.0) * win[k]


@pytest.mark.parametrize("name", ["golden_am_u8", "golden_nfm_s16"])
def test_golden_fixtures_on_the_gpu(cuda, name):
    """The committed golden vectors (tests/golden/*.npz: outputs of the reference's own squelch.cpp / ctcss.cpp / filters.cpp
    objects, written by tests/golden/make_golden.py where /root/reference is mounted) against the CUDA path, with nothing of
    the oracle in between: (1) the stored IQ through the whole engine - bins and decision trace identical, picked-bin IQ
    within 1e-4, audio within 1e-3, counters identical; (2) the stored picked-bin IQ injected behind the channelizer -
    audio, trace and levels bit for bit."""
    import golden_cases
    g = golden_cases.load(name)
    cfg, _ = golden_cases.build(name, with_iq=False)
    nch = len(cfg.devices[0].channels)
    cfg.flags |= abi.FLAG_KEEP_PICKS
    e = Engine(cfg, cuda)
    try:
        for c in range(nch):
            info = e.channel_info(0, c)
            assert info.bin == int(g["bins"][c]) and info.dm_dphi == int(g["dm_dphi"][c])
            assert np.array_equal(np.frombuffer(bytes(info), np.uint8), g["info_raw"][c])
        res = e.run_stream([g["iq"]], chunk_bytes=123_457)[0]
    finally:
        e.close()
    assert res["frames_done"] == int(g["frames"])
    for c in range(nch):
        assert np.array_equal(res["trace"][c], g["trace"][c]), "channel %d: decisions differ from the reference objects'" % c
        assert float(np.abs(res["waveout"][c] - g["waveout"][c]).max()) <= parity.TOL_AUDIO
        got = np.array([[r[c]["axcindicate"], r[c]["bin"], r[c]["open_count"], r[c]["flappy_count"], r[c]["ctcss_count"], r[c]["no_ctcss_count"], r[c]["active_counter"]]
                        for r in res["status"]], np.int64)
        assert np.array_equal(got, g["status_int"][c])
        lv = np.array([[r[c]["signal_level"], r[c]["noise_level"], r[c]["squelch_level"]] for r in res["status"]], np.float32)
        assert np.allclose(lv, g["status_levels"][c], rtol=1e-4, atol=1e-7)
    assert int(((g["trace"] & abi.TRACE_OPEN) != 0).sum()) > 1000
    # (2) the golden picks behind the channelizer: bit-exact.  AFC channels move their bin by what the spectrum says, which
    # injected picks do not carry: compare those that have no AFC.
    cfg2, _ = golden_cases.build(name, with_iq=False)
    e = Engine(cfg2, cuda)
    try:
        picks = np.stack([g["picks"][c] for c in range(nch)], axis=1)  # [frames][C][2]
        waves, traces = [], []
        for lo in range(0, picks.shape[0], 1777):
            e.inject_picks(0, picks[lo:lo + 1777])
            t = e.process()
            r = e.collect(t, 0)
            if r.n_batches:
                waves.append(r.waveout)
                traces.append(r.trace)
    finally:
        e.close()
    wave, trace = np.concatenate(waves, axis=1), np.concatenate(traces, axis=1)
    for c in range(nch):
        if cfg2.devices[0].channels[c].afc:
            continue
        assert np.array_equal(trace[c], g["trace"][c])
        assert np.array_equal(wave[c].view(np.uint32), g["waveout"][c].view(np.uint32)), "channel %d: audio differs from the reference objects' bits" % c


@pytest.mark.parametrize("which", ["mixed", "mixed_quadri", "cfg2", "am_stress"])
def test_demod_bit_exact_against_reference_objects(cuda, which):
    """check_demod_exact with the oracle that drives the reference's OWN squelch.cpp / ctcss.cpp / filters.cpp objects
    (oracle/_ref, compiled from /root/reference/src where it is mounted; the built library travels to the GPU box)."""
    from oracle import ba_oracle
    if not ba_oracle.have_ref():
        pytest.skip("oracle/_ref was not built (it is built only where /root/reference is mounted)")
    if which == "mixed":
        cfg, streams = scenarios.mixed_options(1.2, afc=False)
    elif which == "mixed_quadri":
        cfg, streams = scenarios.mixed_options(1.0, fm_demod=abi.FM_QUADRI_DEMOD, afc=False)
    elif which == "cfg2":
        cfg, streams = scenarios.cfg2_small(8, 1.5)
    else:
        cfg, streams = scenarios.am_stress(2.0)
        cfg.flags = 0
        cfg.max_batches_per_step = 8
    parity.check_demod_exact(cfg, streams, cuda, frames_per_call=2777, ref=True)


def test_end_to_end_against_reference_objects(cuda):
    from oracle import ba_oracle
    if not ba_oracle.have_ref():
        pytest.skip("oracle/_ref was not built (it is built only where /root/reference is mounted)")
    cfg, streams = scenarios.mixed_options(1.2)
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=555_555, ref=True)
    parity.compare_streams(cfg, o, res, min_open=3000)
    cfg, streams = scenarios.afc_walk(1.2)
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=555_555, ref=True)
    parity.compare_streams(cfg, o, res, min_open=2000)


def test_multi_device(cuda):
    cfg, streams = scenarios.multi_device(1.0)
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=300_000)
    parity.compare_streams(cfg, o, res, min_open=1000)


def test_cfg4_wideband_small(cuda):
    """cfg 4's shape at reduced size: cf32, fft 8192, 120 mixed AM/NFM channels, 15.36 Msps."""
    cfg = configs.cfg4(120, sample_rate=15_360_000)
    cfg.flags = abi.FLAG_TRACE
    cfg.max_batches_per_step = 2
    iq = synth.synth(cfg.devices[0], 0.45, 3, gate_on=0.2, gate_off=0.1)
    o, res, _ = parity.run_both(cfg, [iq], cuda, chunk_bytes=2_000_000)
    parity.compare_streams(cfg, o, res, min_open=1000)


def test_ragged_and_empty_input(cuda):
    """Empty submissions, single-byte submissions and a stream shorter than one frame produce nothing and no error;
    feeding the same stream in ragged pieces gives the same result as feeding it at once."""
    cfg, streams = scenarios.cfg1_short(0.35)
    iq = streams[0]
    e = Engine(cfg, cuda)
    e.submit(0, iq[:0])
    t = e.process()
    assert e.collect(t, 0).n_batches == 0
    e.submit(0, iq[:100])
    t = e.process()
    r = e.collect(t, 0)
    assert r.n_batches == 0 and r.frames_done == 0
    e.close()
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=99_991)
    parity.compare_streams(cfg, o, res)
    o2, res2, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=2_000_000)
    assert np.array_equal(res[0]["waveout"], res2[0]["waveout"])


def test_device_resident_stream_matches_host_stream(cuda):
    torch = pytest.importorskip("torch")
    cfg, streams = scenarios.cfg1_short(0.6)
    iq = streams[0]
    o, res, _ = parity.run_both(cfg, streams, cuda)
    e = Engine(cfg, cuda)
    t_iq = torch.from_numpy(iq.copy()).cuda()
    e.attach_device_stream(0, t_iq.data_ptr(), t_iq.numel())
    waves = []
    for lo in range(0, iq.size, 777_777):
        e.advance_device_stream(0, min(777_777, iq.size - lo))
        while True:
            t = e.process()
            r = e.collect(t, 0)
            if not r.n_batches:
                break
            waves.append(r.waveout)
    e.close()
    got = np.concatenate(waves, axis=1)
    assert np.array_equal(got, res[0]["waveout"])


def test_errors(cuda):
    cfg = configs.cfg1()
    cfg.fft_size = 300
    with pytest.raises(EngineError) as ei:
        Engine(cfg, cuda)
    assert ei.value.code == -2  # BA_ERR_BAD_SIZE, as gpu_fft_prepare's -2
    cfg = configs.cfg1()
    cfg.cuda_device = 99
    with pytest.raises(EngineError) as ei:
        Engine(cfg, cuda)
    assert ei.value.code == -1
    cfg = configs.cfg1()
    e = Engine(cfg, cuda)
    big = np.zeros(3_000_000, np.uint8)
    with pytest.raises(EngineError) as ei:
        e.submit(0, big)
    assert ei.value.code == -6  # ring overflow reported (circbuffer_append only counts it)
    e.close()


def test_file_replay_from_a_configuration_file(cuda, tmp_path):
    """Rows f-1/f-2 end to end on the GPU: configuration text -> ba_conf -> engine; IQ files (cs16 and cu8) -> reader
    threads -> pinned input rings -> ba_cuda_process, against the oracle fed the same bytes."""
    conf, cfg, streams = scenarios.file_replay(tmp_path, 1.6)
    parity.check_channel_info(cfg, cuda)
    for chunk in (0, 40_000):
        o, res = parity.run_files(conf, cfg, streams, cuda, chunk_bytes=chunk)
        parity.compare_streams(cfg, o, res, min_open=5000)


@pytest.mark.parametrize("chunk", [300_000, 2_000_000])
def test_mixers(cuda, chunk):
    """Row f-4: mixers summed on the device (K3) behind the demodulator; inputs from three devices arrive unevenly."""
    cfg, streams = scenarios.mixers_on_multi_device(1.5)
    mixed, res, launches = parity.check_mixers(cfg, streams, cuda, chunk)
    assert mixed[1]["right"] is not None and launches > 0


def test_mixer_masked_input(cuda):
    cfg, streams = scenarios.mixers_on_multi_device(1.2)
    streams[1] = streams[1][: len(streams[1]) // 3]
    mixed, res, _ = parity.check_mixers(cfg, streams, cuda, 400_000, masked={0: [1], 1: [1]})
    assert len(mixed[0]["left"]) > len(res[1]["waveout"][0])


@pytest.mark.parametrize("every", [1, 3])
def test_scan_mode(cuda, every):
    """Row f-3: scan mode on the GPU - the freq_t of the channel is switched between batches (ba_cuda_set_freq_idx)."""
    cfg, streams = scenarios.scan_mode(3.0)
    o, res, plan, launches = parity.run_scan(cfg, streams, cuda, every=every, order=[0, 1, 2, 1, 0, 2])
    assert len(plan) >= 6 and len({i for _, i in plan}) == 3
    parity.compare_streams(cfg, o, res, min_open=3000)
    levels = {round(row[0]["squelch_level"], 6) for row in res[0]["status"]}
    assert len(levels) > 3  # the manual-level frequency and the automatic ones both ran


def test_cfg5_full_size_replicas_and_oracle(cuda):
    """BASELINE cfg 5 at its full size on one GPU: 512 inputs x 2.56 Msps u8, fft 512, 16 AM channels each (8192 channels, the
    plain demodulator).  Size-independent properties: inputs that carry the same bytes under the same channel offsets
    (every 8th input) give bit-identical audio and status, whichever SM and slot they ran on; one input of each of
    the 8 kinds is compared with the oracle.  Inputs are device-resident, as in bench.py."""
    torch = pytest.importorskip("torch")
    from oracle.ba_oracle import Oracle
    cfg = configs.cfg5(512, 512)
    cfg.max_batches_per_step = 4
    seconds = 1.3
    tmpl = [synth.synth(cfg.devices[k], seconds, k, gate_on=0.35, gate_off=0.12) for k in range(8)]
    dev_tmpl = [torch.from_numpy(t.copy()).cuda() for t in tmpl]
    e = Engine(cfg, cuda)
    keep = []
    try:
        for i in range(512):
            t = dev_tmpl[i % 8].clone()  # a private copy per input, as separate dongles would have
            keep.append(t)
            e.attach_device_stream(i, t.data_ptr(), t.numel())
        waves = [[] for _ in range(512)]
        stats = [[] for _ in range(512)]
        total = tmpl[0].size
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
        launches = e.launch_count()
    finally:
        e.close()
    assert launches > 0
    full = [np.concatenate(w, axis=1) for w in waves]
    st = [np.concatenate(x, axis=0) for x in stats]
    n_batches = full[0].shape[1] // cfg.wave_batch
    assert n_batches == cfg.batches_for(0, total) and n_batches >= 9
    for i in range(8, 512):
        assert np.array_equal(full[i].view(np.uint32), full[i % 8].view(np.uint32)), "input %d differs from input %d" % (i, i % 8)
        assert np.array_equal(st[i], st[i % 8]), "status of input %d differs from input %d" % (i, i % 8)
    sub = abi.EngineCfg(fft_size=512, wave_rate=8000, devices=[cfg.devices[k] for k in range(8)])
    o = Oracle(sub)
    opened = 0
    for k in range(8):
        o.feed(k, tmpl[k])
        for c in range(16):
            wo = o.waveout(k, c)
            assert len(wo) == full[k].shape[1]
            assert float(np.abs(wo - full[k][c]).max()) <= parity.TOL_AUDIO
            so = o.status(k, c)
            for b, s_ in enumerate(so):
                assert int(st[k][b, c, 0].view(np.int32)) == s_.axcindicate and int(st[k][b, c, 5]) == s_.open_count
            opened += sum(1 for s_ in so if s_.axcindicate != abi.NO_SIGNAL)
    assert opened > 100


def test_cfg4_full_size(cuda):
    """BASELINE cfg 4 at its full size: one 61.44 Msps cf32 stream, fft 8192, 2000 mixed AM/NFM channels (250 with CTCSS and
    notch).  Squelch decisions identical, audio within 1e-3, for every channel."""
    cfg = configs.cfg4()
    cfg.flags = abi.FLAG_TRACE
    cfg.max_batches_per_step = 2
    torch = pytest.importorskip("torch")
    n = int(0.3 * cfg.devices[0].sample_rate)  # 2000 carriers x 18 M samples: synthesised on the GPU, checked on the CPU
    iq = synth.synth_torch(cfg.devices[0], n, 5, torch.device("cuda", 0), gate_on=0.12, gate_off=0.06).cpu().numpy()
    torch.cuda.empty_cache()
    o, res, _ = parity.run_both(cfg, [iq], cuda, chunk_bytes=64_000_000)
    parity.compare_streams(cfg, o, res, min_open=100_000)


def test_results_on_device_equal_results_on_host(cuda):
    """BA_FLAG_RESULTS_ON_DEVICE: the audio stays in HBM (device pointers in ba_step_out) - the same bytes a host copy gives."""
    import ctypes as C
    from boondock_airband_b200.engine import device_to_host
    cfg, streams = scenarios.cfg1_short(0.6)
    cfg.flags = 0
    o, res, _ = parity.run_both(cfg, streams, cuda, chunk_bytes=500_000)
    cfg.flags = abi.FLAG_RESULTS_ON_DEVICE
    e = Engine(cfg, cuda)
    waves = []
    try:
        iq = streams[0]
        for lo in range(0, iq.size, 500_000):
            e.submit(0, iq[lo:lo + 500_000])
            t = e.process()
            out = e.collect_raw(t, 0)
            if out.n_batches:
                n = out.n_batches * out.wave_batch
                rows = []
                for c in range(out.channel_count):
                    ptr = C.cast(out.waveout, C.c_void_p).value + 4 * c * out.wave_stride
                    rows.append(np.frombuffer(device_to_host(ptr, 4 * n), np.float32))
                waves.append(np.stack(rows))
                assert out.status[0].bin == e.channel_info(0, 0).bin  # status still arrives on the host
    finally:
        e.close()
    got = np.concatenate(waves, axis=1)
    assert np.array_equal(got.view(np.uint32), res[0]["waveout"].view(np.uint32))


def test_two_engines_on_two_gpus_in_one_process(cuda):
    """One engine per GPU inside one process (boondock_airband.cpp:1088-1122: one demod thread per device).  Skipped on a box
    with a single GPU."""
    from boondock_airband_b200 import engine as eng_mod
    if int(eng_mod.load_library().ba_cuda_visible_devices()) < 2:
        pytest.skip("needs two GPUs")
    cfg0, streams = scenarios.cfg1_short(0.9)
    cfg1, _ = scenarios.cfg1_short(0.9)
    cfg1.cuda_device = 1
    e0, e1 = Engine(cfg0, cuda), Engine(cfg1, cuda)
    try:
        r1 = e1.run_stream(streams, chunk_bytes=500_000)
        r0 = e0.run_stream(streams, chunk_bytes=700_001)
    finally:
        e0.close()
        e1.close()
    for c in range(len(cfg0.devices[0].channels)):
        assert np.array_equal(r0[0]["waveout"][c].view(np.uint32), r1[0]["waveout"][c].view(np.uint32))
    assert r0[0]["frames_done"] == r1[0]["frames_done"] > 0


@pytest.mark.parametrize("which", ["cfg1", "mixed", "multi"])
def test_skip_silent_rows(cuda, which):
    """BA_FLAG_SKIP_SILENT_ROWS: the packed rows and their map, put back together, are the audio of a run without the flag bit for
    bit (plain and general channels, several inputs of different rates), and silent rows were in fact left out of the copy."""
    if which == "cfg1":
        cfg, streams = scenarios.cfg1_short(1.9)
        cfg_b, _ = scenarios.cfg1_short(1.9)
    elif which == "mixed":
        cfg, streams = scenarios.mixed_options(1.5)
        cfg_b, _ = scenarios.mixed_options(1.5)
    else:
        cfg, streams = scenarios.multi_device(0.9)
        cfg_b, _ = scenarios.multi_device(0.9)
    cfg.flags &= ~abi.FLAG_TRACE
    cfg_b.flags = (cfg_b.flags & ~abi.FLAG_TRACE) | abi.FLAG_SKIP_SILENT_ROWS
    e = Engine(cfg, cuda)
    want = e.run_stream(streams, chunk_bytes=600_000)
    e.close()
    e = Engine(cfg_b, cuda)
    got = e.run_stream(streams, chunk_bytes=450_001)
    e.close()
    assert sum(g["rows_skipped"] for g in got) > 0
    for d in range(len(cfg.devices)):
        for c in range(len(cfg.devices[d].channels)):
            assert np.array_equal(want[d]["waveout"][c].view(np.uint32), got[d]["waveout"][c].view(np.uint32)), (d, c)
        assert got[d]["status"] == want[d]["status"]
        if want[d]["iq_out"] is not None:
            assert np.array_equal(want[d]["iq_out"], got[d]["iq_out"])
