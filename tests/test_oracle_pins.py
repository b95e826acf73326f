"""Pins the CPU oracle (oracle/dsp_restated.h + oracle.cpp) before anything is compared against it:
  1. the behavioural scenarios of the reference's own unit tests (test_squelch.cpp:56-281, test_ctcss.cpp:122-155,
     test_filters.cpp:33-41), replayed against the restated classes;
  2. the committed golden fixtures (tests/golden/*.npz), which were produced by the reference's own squelch.cpp /
     ctcss.cpp / filters.cpp compiled unmodified (tests/golden/make_golden.py);
  3. where oracle/_ref exists, a bit-for-bit comparison of the restatement with that reference build on fresh inputs.
The FFT itself is outside the reference tree (FFTW, unpinned): it is bounded against a float64 DFT."""
import math
import os

import numpy as np
import pytest

from boondock_airband_b200 import abi, configs, synth
from boondock_airband_b200.abi import ChannelCfg, DeviceCfg, EngineCfg

import golden_cases

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NOISE, SIGNAL = 0.05, 0.75
STANDARD_TONES = [67.0, 69.3, 71.9, 74.4, 77.0, 79.7, 82.5, 85.4, 88.5, 91.5, 94.8, 97.4, 100.0, 103.5, 107.2, 110.9, 114.8, 118.8, 123.0, 127.3, 131.8, 136.5,
                  141.3, 146.2, 150.0, 151.4, 156.7, 159.8, 162.2, 165.5, 167.9, 171.3, 173.8, 177.3, 179.9, 183.5, 186.2, 189.9, 192.8, 196.6, 199.5, 203.5, 206.5,
                  210.7, 218.1, 225.7, 229.1, 233.6, 241.8, 250.3, 254.1]


@pytest.fixture(scope="module")
def orc(oracle_built):
    return oracle_built


def builds(orc):
    return [False, True] if orc.have_ref() else [False]


def settle_noise_floor(p):
    """send_samples_for_noise_floor, test_squelch.cpp:39-46"""
    n = 0
    while p.query()["noise_level"] > 1.01 * NOISE:
        p.raw(NOISE)
        n += 1
        assert n < 100000
    q = p.query()
    assert q["noise_level"] <= 1.01 * NOISE and SIGNAL > q["squelch_level"]


def tone_source(freq, rate, ampl=0.2):
    """Tone::get_sample, generate_signal.cpp:34-37 (the counter starts at 1)"""
    n = 0
    while True:
        n += 1
        yield np.float32(ampl * math.sin(2 * math.pi * n * freq / rate))


@pytest.mark.parametrize("ref", [False, True])
def test_squelch_reference_scenarios(orc, ref):
    if ref and not orc.have_ref():
        pytest.skip("oracle/_ref is built only where /root/reference is mounted")
    P = lambda: orc.SquelchProbe(ref=ref)  # noqa: E731
    # default_object
    assert P().query()["open_count"] == 0
    # noise_floor (test_squelch.cpp:56-79)
    p = P()
    assert p.query()["noise_level"] > 10 * NOISE
    this = p.query()["noise_level"]
    while True:
        last = this
        for _ in range(25):
            p.raw(NOISE)
        this = p.query()["noise_level"]
        assert this <= last
        if this == last:
            break
    assert p.query()["noise_level"] < 1.01 * NOISE
    # normal_operation (:81-109)
    p = P()
    settle_noise_floor(p)
    for _ in range(500):
        if p.query()["is_open"]:
            break
        p.raw(SIGNAL)
    q = p.query()
    assert q["is_open"] and q["should_process_audio"]
    for _ in range(1000):
        p.raw(SIGNAL)
    assert p.query()["is_open"]
    for _ in range(100):
        if not p.query()["is_open"]:
            break
        p.raw(NOISE)
    q = p.query()
    assert not q["is_open"] and not q["should_process_audio"]
    # dead_spot (:111-143)
    p = P()
    settle_noise_floor(p)
    for _ in range(500):
        if p.query()["is_open"]:
            break
        p.raw(SIGNAL)
    for _ in range(1000):
        p.raw(SIGNAL)
    for _ in range(50):
        p.raw(NOISE)
        q = p.query()
        assert q["is_open"] and q["should_process_audio"]
    for _ in range(1000):
        p.raw(SIGNAL)
        assert p.query()["is_open"]
    # should_process_audio (:145-165)
    p = P()
    settle_noise_floor(p)
    for _ in range(500):
        if p.query()["is_open"]:
            break
        assert not p.query()["should_process_audio"]
        p.raw(SIGNAL)
    assert p.query()["is_open"] and p.query()["should_process_audio"]
    for _ in range(100):
        if not p.query()["is_open"]:
            break
        assert p.query()["should_process_audio"]
        p.raw(NOISE)
    assert not p.query()["is_open"] and not p.query()["should_process_audio"]


@pytest.mark.parametrize("ref", [False, True])
@pytest.mark.parametrize("case", ["good", "wrong", "close"])
def test_squelch_ctcss_scenarios(orc, ref, case):
    """good_ctcss / wrong_ctcss / close_ctcss, test_squelch.cpp:167-281 (fs 8000)."""
    if ref and not orc.have_ref():
        pytest.skip("oracle/_ref is built only where /root/reference is mounted")
    rate = 8000.0
    actual, expected = {"good": (5, 5), "wrong": (0, 7), "close": (5, 7)}[case]
    p = orc.SquelchProbe(ref=ref)
    p.set_ctcss(STANDARD_TONES[expected], rate)
    settle_noise_floor(p)
    src = tone_source(STANDARD_TONES[actual], rate)
    for _ in range(500):
        if p.query()["should_process_audio"]:
            break
        p.raw(SIGNAL)
    q = p.query()
    assert q["should_process_audio"] and not q["is_open"]
    long_run = 20000  # the reference runs 100 000; the decision pattern repeats every 3200 samples
    if case == "good":
        for _ in range(500):
            if p.query()["is_open"]:
                break
            p.audio(float(next(src)))
            p.raw(SIGNAL)
        assert p.query()["is_open"]
        for _ in range(long_run):
            p.audio(float(next(src)))
            p.raw(SIGNAL)
        q = p.query()
        assert q["is_open"] and q["should_process_audio"]
        assert q["ctcss_count"] > 0 and q["no_ctcss_count"] == 0
    elif case == "wrong":
        for i in range(long_run):
            p.audio(float(next(src)))
            p.raw(SIGNAL)
            if i % 97 == 0:
                q = p.query()
                assert q["should_process_audio"] and not q["is_open"]
        q = p.query()
        assert q["ctcss_count"] == 0 and q["no_ctcss_count"] > 0
    else:
        for _ in range(500):
            if p.query()["is_open"]:
                break
            p.audio(float(next(src)))
            p.raw(SIGNAL)
        assert p.query()["is_open"]
        for _ in range(3000):
            if not p.query()["is_open"]:
                break
            p.audio(float(next(src)))
            p.raw(SIGNAL)
        assert not p.query()["is_open"]
        for i in range(long_run):
            p.audio(float(next(src)))
            p.raw(SIGNAL)
            if i % 97 == 0:
                q = p.query()
                assert q["should_process_audio"] and not q["is_open"]
        q = p.query()
        assert q["ctcss_count"] == 0 and q["no_ctcss_count"] > 0


@pytest.mark.parametrize("ref", [False, True])
def test_ctcss_reference_scenarios(orc, ref):
    """no_signal / has_tone / has_non_standard_tone / has_each_standard_tone, test_ctcss.cpp:122-155, seeded noise."""
    if ref and not orc.have_ref():
        pytest.skip("oracle/_ref is built only where /root/reference is mounted")
    rate, window = 8000.0, 3200
    rng = np.random.default_rng(7)
    silence = np.zeros(window, np.float32)
    for det in STANDARD_TONES:
        tone, enough = orc.ctcss_run(det, rate, window, silence, ref=ref)
        assert enough and not tone
    t = np.arange(1, window + 1)

    def check(freq):
        x = (0.2 * np.sin(2 * np.pi * t * freq / rate) + 0.2 * 0.1 * rng.standard_normal(window)).astype(np.float32)
        for det in STANDARD_TONES:
            if abs(det - freq) < 5:
                continue
            tone, enough = orc.ctcss_run(det, rate, window, x, ref=ref)
            assert enough and not tone, (freq, det)
        tone, enough = orc.ctcss_run(freq, rate, window, x, ref=ref)
        assert enough and tone, freq

    check(STANDARD_TONES[0])
    check((STANDARD_TONES[0] + STANDARD_TONES[0]) / 2)
    for f in STANDARD_TONES:
        check(f)


def test_filters_default_disabled(orc):
    """test_filters.cpp:33-41: a filter constructed without a frequency passes samples through."""
    x = np.linspace(-1, 1, 50).astype(np.float32)
    y, _ = orc.notch_run(0.0, 8000.0, 10.0, x)
    assert np.array_equal(x, y)
    z = (x + 1j * x[::-1]).astype(np.complex64)
    assert np.array_equal(orc.lowpass_run(0.0, 8000.0, z).astype(np.complex64), z)


def test_filter_responses(orc):
    """The reference has no response test; pin the obvious ones: the notch nulls its frequency and passes the rest,
    the Bessel low-pass has unity DC gain and attenuates beyond the cut-off."""
    rate = 16000.0
    n = np.arange(8000)
    for hz, expect_low in ((100.0, True), (1000.0, False)):
        x = np.sin(2 * np.pi * hz * n / rate).astype(np.float32)
        y, _ = orc.notch_run(100.0, rate, 10.0, x)
        amp = float(np.abs(y[4000:]).max())
        assert (amp < 0.05) if expect_low else (0.9 < amp < 1.1), (hz, amp)
    z = np.ones(4000, np.complex64)
    y = orc.lowpass_run(6250.0, rate, z)
    assert abs(y[-1] - 1.0) < 1e-3
    z = np.exp(2j * np.pi * 7900.0 * np.arange(4000) / rate).astype(np.complex64)
    y = orc.lowpass_run(2000.0, rate, z)
    assert float(np.abs(y[2000:]).max()) < 0.1


def test_golden_dsp_objects(orc):
    """The restated Squelch / CTCSS / filters reproduce, bit for bit, what the reference's own objects produced."""
    g = np.load(os.path.join(GOLD, "dsp_objects.npz"))
    raw, filt, audio = g["sq_raw"], g["sq_filtered"], g["sq_audio"]
    for tag, kw in (("plain", {}), ("filtered", dict(filtered=filt)), ("ctcss", dict(audio=audio, ctcss=100.0)), ("manual", dict(level=0.3))):
        p = orc.SquelchProbe()
        if "ctcss" in kw:
            p.set_ctcss(kw["ctcss"], 8000.0)
        if "level" in kw:
            p.set_level(kw["level"])
        st, lv = p.run(raw, kw.get("filtered"), kw.get("audio"), want_levels=True)
        assert np.array_equal(st, g["sq_states_" + tag]), tag
        assert np.array_equal(lv.view(np.uint32), g["sq_levels_" + tag].view(np.uint32)), tag
        q = p.query()
        assert [q["open_count"], q["flappy_count"], q["ctcss_count"], q["no_ctcss_count"]] == list(g["sq_counts_" + tag]), tag
    # the stimulus exercises every state, flapping and both CTCSS outcomes
    assert set(np.unique(g["sq_states_plain"] & 7)) == {0, 1, 2, 3, 4}
    assert g["sq_counts_plain"][1] > 0
    tones, sig, dec = g["ctcss_tones"], g["ctcss_signals"], g["ctcss_decisions"]
    for i in range(0, tones.size, 3):
        for j in range(tones.size):
            tone, enough = orc.ctcss_run(float(tones[j]), 8000.0, 3200, sig[i])
            assert enough and int(tone) == int(dec[i, j]), (i, j)
    y, _ = orc.notch_run(100.0, 16000.0, 10.0, g["notch_in"])
    assert np.array_equal(y.view(np.uint32), g["notch_out"].view(np.uint32))
    z = orc.lowpass_run(6250.0, 16000.0, g["lp_in"]).astype(np.complex64)
    assert np.array_equal(z.view(np.uint32), g["lp_out"].view(np.uint32))


@pytest.mark.parametrize("name", golden_cases.NAMES)
def test_golden_pipeline(orc, name):
    """The restated loop + restated classes reproduce the reference-built oracle's committed outputs bit for bit."""
    g = golden_cases.load(name)
    cfg, _ = golden_cases.build(name, with_iq=False)
    o = orc.Oracle(cfg)
    o.feed(0, g["iq"])
    assert o.frames(0) == int(g["frames"]) and o.batches(0) == int(g["batches"])
    nch = len(cfg.devices[0].channels)
    for c in range(nch):
        info = o.channel_info(0, c)
        assert info.bin == int(g["bins"][c]) and info.dm_dphi == int(g["dm_dphi"][c])
        assert np.array_equal(np.frombuffer(bytes(info), np.uint8), g["info_raw"][c])
        assert np.array_equal(o.waveout(0, c).view(np.uint32), g["waveout"][c].view(np.uint32))
        assert np.array_equal(o.trace(0, c), g["trace"][c])
        assert np.array_equal(o.picks(0, c).view(np.uint32), g["picks"][c].view(np.uint32))
        st = o.status(0, c)
        got = np.array([[s.axcindicate, s.bin, s.open_count, s.flappy_count, s.ctcss_count, s.no_ctcss_count, s.active_counter] for s in st], np.int64)
        assert np.array_equal(got, g["status_int"][c])
    if "iq_out" in g:
        for k, c in enumerate(g["iq_channels"]):
            assert np.array_equal(o.iq_out(0, int(c)).view(np.uint32), g["iq_out"][k].view(np.uint32))


def test_restated_equals_reference_build(orc):
    """Fresh inputs, every option: the restatement and the reference's own objects give identical bits."""
    if not orc.have_ref():
        pytest.skip("oracle/_ref is built only where /root/reference is mounted")
    import scenarios
    for cfg, streams in (scenarios.mixed_options(0.6), scenarios.mixed_options(0.5, fm_demod=abi.FM_QUADRI_DEMOD), scenarios.cfg2_small(4, 1.0), scenarios.multi_device(0.4)):
        a, b = orc.Oracle(cfg), orc.Oracle(cfg, ref=True)
        for d, s in enumerate(streams):
            a.feed(d, s)
            b.feed(d, s)
        for d, dev in enumerate(cfg.devices):
            for c in range(len(dev.channels)):
                assert bytes(a.channel_info(d, c)) == bytes(b.channel_info(d, c))
                assert np.array_equal(a.waveout(d, c).view(np.uint32), b.waveout(d, c).view(np.uint32))
                assert np.array_equal(a.trace(d, c), b.trace(d, c))
                sa, sb = a.status(d, c), b.status(d, c)
                assert [bytes(x) for x in sa] == [bytes(x) for x in sb]


@pytest.mark.parametrize("name", sorted(golden_cases.digest_scenarios()))
def test_oracle_reproduces_recorded_outputs(orc, name):
    """The scenarios of test_restated_equals_reference_build and of the GPU tests against the reference objects (FM quadri
    demodulation, cfg2's CTCSS and notch, several inputs, the AGC clip and flapping of am_stress, the AFC walk): the oracle's
    outputs, bit for bit, against the digests in golden/oracle_digests.json, and the reference-built oracle's too where it exists."""
    import json
    with open(os.path.join(GOLD, "oracle_digests.json")) as f:
        want = json.load(f)[name]
    cfg, streams = golden_cases.digest_scenarios()[name]()
    for ref in builds(orc):
        got = golden_cases.oracle_digests(orc.Oracle, cfg, streams, ref=ref)
        assert got["inputs"] == want["inputs"], "the scenario's synthesised input is not the recorded one"
        for key in sorted(want["channels"]):
            assert got["channels"][key] == want["channels"][key], (ref, key)
        assert got == want


def test_oracle_fft_against_float64_dft(orc):
    """FFT parity is unpinned by the reference (FFTW is not in its tree): the oracle's float FFT stays within 1e-6 of the exact DFT."""
    rng = np.random.default_rng(3)
    for n in (256, 512, 1024, 2048, 4096, 8192):
        dev = DeviceCfg(sample_rate=2_400_000, centerfreq=100_000_000, sample_format="f32", channels=[ChannelCfg(freq=100_100_000)])
        cfg = EngineCfg(fft_size=n, wave_rate=16000, devices=[dev])
        iq = (rng.standard_normal(2 * (n + 150 * 3)) * 0.3).astype(np.float32)
        o = orc.Oracle(cfg)
        fi, fo = o.debug_frames(0, iq, 4)
        ref = np.fft.fft(fi[..., 0].astype(np.float64) + 1j * fi[..., 1], axis=1)
        got = fo[..., 0].astype(np.float64) + 1j * fo[..., 1]
        assert float(np.abs(got - ref).max() / np.abs(ref).max()) < 1e-6


def test_bin_and_phase_formulas(orc):
    """Known answers worked out by hand from config.cpp:669-670 and :682-715 (SURVEY.md section 8a, row A2)."""
    cfg = configs.cfg1()
    o = orc.Oracle(cfg)
    assert o.channel_info(0, 2).bin == 411   # 119.5 MHz at centre 120.0, 2.56 Msps, 512 bins
    assert o.channel_info(0, 4).bin == 44    # 120.225 MHz
    dev = DeviceCfg(sample_rate=2_400_000, centerfreq=162_482_000, sample_format="s16", channels=[ChannelCfg(freq=162_400_000, modulation="nfm")])
    o = orc.Oracle(EngineCfg(fft_size=1024, wave_rate=16000, devices=[dev]))
    info = o.channel_info(0, 0)
    assert info.bin == 989                   # Fs / N is an integer division: 2343, not 2343.75
    # dm_dphi: (freq - centre) / WAVE_RATE, fractional part, scaled to 24 bits; -82 kHz / 16 kHz = -5.125 -> -0.125 * 2^24
    assert info.dm_dphi == (int(-0.125 * (1 << 24)) & 0xFFFFFFFF)


def _rn32(x):
    """Round an exact rational to the nearest IEEE binary32 (ties to even); normal range only. Returns a Fraction."""
    from fractions import Fraction
    if x == 0:
        return Fraction(0)
    s = -1 if x < 0 else 1
    a = abs(x)
    e = 0
    while a >= 2:
        a /= 2
        e += 1
    while a < 1:
        a *= 2
        e -= 1
    assert -126 <= e <= 127
    m = a * (1 << 23)  # in [2^23, 2^24)
    lo = m.numerator // m.denominator
    rem = m - lo
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and (lo & 1)):
        lo += 1
    return s * Fraction(lo, 1 << 23) * (Fraction(2) ** e)


def test_u8_level_formula():
    """K1 forms the u8 level (i - 127.5f) / 127.5f (boondock_airband.cpp:341-343) without a division:
    fma(a, r_hi, RN(a * r_lo)) with a = i - 127.5 and a two-float reciprocal of 127.5 (channelize.cu: level_u8 / sample_u8).
    Exact rational arithmetic: for all 256 codes the result equals the correctly rounded quotient, which is what the
    reference's float division produces."""
    from fractions import Fraction
    r_hi = Fraction(float.fromhex("0x1.010102p-7"))
    r_lo = Fraction(float.fromhex("-0x1.fdfdfep-32"))
    assert _rn32(r_hi) == r_hi and _rn32(r_lo) == r_lo  # both are binary32 values
    for code in range(256):
        a = Fraction(2 * code - 255, 2)          # i - 127.5, exact in binary32
        assert _rn32(a) == a
        want = _rn32(a / Fraction(255, 2))       # IEEE division: the correctly rounded quotient
        got = _rn32(a * r_hi + _rn32(a * r_lo))  # fma rounds once; the inner product is rounded separately
        assert got == want, code
        # and the table the reference fills is what numpy's float32 division gives
        assert float(want) == float(np.float32(code - 127.5) / np.float32(127.5))


def _mix_with_restatement(orc, ampfactor, balance, x, has_signal):
    """oracle/ba_oracle.py: mix_reference on explicit batches (input j = channel 0 of a pretend device j)."""
    from boondock_airband_b200.abi import MixerCfg, MixerInputCfg
    n_b, n_in, B = x.shape
    cfg = EngineCfg(fft_size=512, wave_rate=8 * B, devices=[])
    mixer = MixerCfg("pin", [MixerInputCfg(j, 0, ampfactor=float(ampfactor[j]), balance=float(balance[j])) for j in range(n_in)])

    class St:
        def __init__(self, a):
            self.axcindicate = a
    wave = lambda d, c: np.ascontiguousarray(x[:, d, :]).reshape(-1)
    stat = lambda d, c: [St(abi.SIGNAL if has_signal[k, d] else abi.NO_SIGNAL) for k in range(n_b)]
    return orc.mix_reference(cfg, wave, stat, mixer)


def test_mixer_restatement_against_a_run_of_the_reference_mixer(orc):
    """tests/golden/golden_mixer.npz was produced by the reference's own mixer.cpp (mixer_connect_input, mixer_put_samples,
    mixer_thread; tests/golden/make_golden_mixer.py).  The restated summing the device-side mixer is compared with
    (oracle/ba_oracle.py: mix_reference) reproduces it bit for bit: multipliers ampfactor * min(1, 1 -/+ balance), inputs without
    signal skipped, a zero multiplier skipped, stereo as soon as one balance is non-zero, SIGNAL iff any input had signal."""
    g = np.load(os.path.join(GOLD, "golden_mixer.npz"))
    left, right, sig = _mix_with_restatement(orc, g["ampfactor"], g["balance"], g["x"], g["has_signal"])
    assert int(g["stereo"]) == 1 and right is not None
    assert np.array_equal(left.view(np.uint32), g["left"].reshape(-1).view(np.uint32))
    assert np.array_equal(right.view(np.uint32), g["right"].reshape(-1).view(np.uint32))
    want = np.where(g["axcindicate"] == ord("*"), abi.SIGNAL, abi.NO_SIGNAL)
    assert list(sig) == list(want)
    assert (g["axcindicate"] == ord(" ")).any() and (g["left"][2] == 0).all()  # the batch in which nobody had signal


def test_reference_mixer_reproduces_the_fixture(orc):
    """Where the reference tree is mounted: the committed fixture is what its mixer produces today."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_mixer", os.path.join(GOLD, "make_golden_mixer.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    if not (orc.have_ref() and os.path.exists(mg.LIB)):
        pytest.skip("oracle/_ref/libba_mixer_ref.so is not built (needs /root/reference)")
    a, b, x, s = mg.case()
    left, right, axc, stereo = mg.run_reference(a, b, x, s)
    g = np.load(os.path.join(GOLD, "golden_mixer.npz"))
    assert np.array_equal(left, g["left"]) and np.array_equal(right, g["right"]) and np.array_equal(axc, g["axcindicate"]) and stereo == int(g["stereo"])
