"""Rows f-2 and f-1 of SURVEY.md section 8, on the CPU: the configuration front-end (libconfig-subset reader + the rules of
parse_devices()/parse_channels(), src/config.cpp:298-836) and the file input (src/input-file.cpp:35-181), through
libba_host.so.  The expected values are the reference's own arithmetic restated in Python next to each assertion."""
import ctypes as C
import math
import os
import re
import subprocess
import time

import numpy as np
import pytest

from boondock_airband_b200 import abi, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ba_host.h")
REF_CONFIGS = "/root/reference/config"


@pytest.fixture(scope="module", autouse=True)
def built():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "boondock_airband_b200", "csrc"), "../libba_host.so"], stdout=subprocess.DEVNULL)


OUT = 'outputs: ( { type = "file"; directory = "/tmp"; filename_template = "x"; } );'

# written for this test in the style of config/basic_multichannel.conf
BASIC = """
# comment
fft_size = 512;
devices:
({
  type = "rtlsdr";
  index = 0;
  gain = 25;
  centerfreq = 120.0;       // float: MHz
  correction = 80;
  channels:
  (
    { freq = 119.5; %(o)s },
    { freq = 120225000; label = "int Hz"; %(o)s },
    { freq = "119.15M"; afc = 2; ampfactor = 2.5; squelch_threshold = -40; %(o)s },
    { freq = 121.0; disable = true; %(o)s },
    { freq = 120.8; squelch_snr_threshold = 6; notch = 1000.0; notch_q = 4.0; %(o)s }
  );
 }
);
""" % {"o": OUT}


def test_basic_multichannel_model():
    c = host.parse_text(BASIC)
    cfg = c.cfg
    assert cfg.fft_size == 512 and cfg.wave_rate == 8000 and len(cfg.devices) == 1
    d = cfg.devices[0]
    # rtlsdr_input_new presets (input-rtlsdr.cpp:244-247)
    assert (d.sample_format, d.sample_rate, d.fullscale) == ("u8", 2560000, 126.5)
    assert d.centerfreq == int(120.0 * 1e6)
    ch = d.channels
    assert [c.source_index(0, k) for k in range(len(ch))] == [0, 1, 2, 4] and c.source_index(0, 4) == -1
    assert ch[0].freq == int(119.5 * 1e6) and ch[1].freq == 120225000 and ch[2].freq == int(119.15 * 1e6)
    assert (ch[2].afc, ch[2].ampfactor, ch[2].squelch_threshold) == (2, 2.5, -40)
    assert ch[0].squelch_snr_threshold == -1.0 and ch[3].squelch_snr_threshold == 6.0
    assert (ch[3].notch, ch[3].notch_q) == (1000.0, 4.0)
    assert all(x.modulation == "am" and x.bandwidth == 0 and not x.has_iq_outputs for x in ch)
    assert c.setting(0, "gain") == "25" and c.setting(0, "type") == "rtlsdr" and c.setting(0, "nope") is None
    assert c.warnings == []


def test_float_megahertz_is_truncated_like_the_reference():
    """parse_anynum2int: (int)((double)f * 1e6) truncates, so 128.2 MHz is 128199999 Hz (config.cpp:303)."""
    freqs = [162.4, 162.425, 162.55, 128.2, 128.075, 0.1 + 0.2]
    text = 'devices: ({ type = "rtlsdr"; centerfreq = 162.482; sample_rate = 2.4; channels: (%s); });' % ",".join(
        "{ freq = %r; %s }" % (f, OUT) for f in freqs)
    c = host.parse_text(text, 8000)
    assert [x.freq for x in c.cfg.devices[0].channels] == [int(f * 1e6) for f in freqs]
    assert int(128.2 * 1e6) == 128199999  # the quirk this test is about
    assert c.cfg.devices[0].sample_rate == int(2.4 * 1e6) and c.cfg.devices[0].centerfreq == int(162.482 * 1e6)
    assert any("outside of SDR operating bandwidth" in w for w in c.warnings)  # 0.3 MHz is far off


def test_suffixed_strings_follow_atofs():
    """atofs(): trailing k/M/G multiply (util.cpp:130-155)."""
    text = 'devices: ({ type = "rtlsdr"; centerfreq = "120M"; sample_rate = "2400k"; channels: ({ freq = "0.1195G"; bandwidth = "12.5k"; %s }); });' % OUT
    d = host.parse_text(text, 16000).cfg.devices[0]
    assert d.centerfreq == 120000000 and d.sample_rate == 2400000
    assert d.channels[0].freq == int(1e3 * 1e3 * 1e3 * 0.1195) and d.channels[0].bandwidth == int(1e3 * 12.5)


NFM = """
fft_size = 1024;
multiple_demod_threads = true;
tau = 75;
devices: ({
  type = "soapysdr"; device_string = "driver=x"; sample_format = "CS16";
  centerfreq = 162482000; sample_rate = 2400000;
  tau = 530;
  channels: (
    { freq = 162400000; modulation = "nfm"; bandwidth = 5000; ampfactor = 2.00; squelch_snr_threshold = 0.00; ctcss = 100.0; notch = 100.0; %(o)s },
    { freq = 162425000; modulation = "nfm"; tau = 0; outputs: ( { type = "rawfile"; directory = "/tmp"; filename_template = "iq"; } ); },
    { freq = 162450000; modulation = "am"; %(o)s }
  );
});
""" % {"o": OUT}


def test_nfm_build_is_inferred_and_options_carry():
    c = host.parse_text(NFM)
    cfg = c.cfg
    assert cfg.wave_rate == 16000 and cfg.fft_size == 1024 and c.multiple_demod_threads
    d = cfg.devices[0]
    assert (d.sample_format, d.bytes_per_sample, d.fullscale, d.tau) == ("s16", 2, 32766.5, 530)
    a, b, am = d.channels
    assert (a.modulation, a.bandwidth, a.ampfactor, a.squelch_snr_threshold, a.ctcss, a.notch, a.notch_q, a.tau) == ("nfm", 5000, 2.0, 0.0, 100.0, 100.0, 10.0, -1)
    assert (b.modulation, b.tau, b.has_iq_outputs) == ("nfm", 0, True)
    assert am.modulation == "am"
    # the AM-only build of the reference does not know "nfm" (config.cpp:341-352)
    with pytest.raises(host.ConfigError, match="unknown modulation"):
        host.parse_text(NFM, 8000)


def test_root_tau_is_the_default_of_devices_without_their_own():
    text = 'tau = 75; devices: ({ type = "rtlsdr"; centerfreq = 100.0; channels: ({ freq = 100.1; modulation = "nfm"; %s }); });' % OUT
    assert host.parse_text(text).cfg.devices[0].tau == 75
    assert host.parse_text(text.replace("tau = 75; ", "")).cfg.devices[0].tau == -1


def one_channel(body, wave_rate=16000, dev_extra=""):
    return host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 120.0; %s channels: ({ freq = 120.1; %s %s }); });' % (dev_extra, body, OUT), wave_rate)


@pytest.mark.parametrize("body,message", [
    ("lowpass = 50;", r"lowpass \(50\) must be greater than or equal to highpass \(100\)"),
    ('modulation = "fm";', "unknown modulation"),
    ("squelch_threshold = 5;", "squelch_threshold must be less than or equal to 0"),
    ("squelch_threshold = -40.0;", "Invalid value for squelch_threshold"),
    ("squelch_snr_threshold = -3;", "squelch_snr_threshold must be greater than or equal to 0"),
    ('squelch_snr_threshold = "x";', "Invalid value for squelch_snr_threshold"),
    ("notch = 100;", "notch should be an float"),
    ("notch = 100.0; notch_q = 5;", "notch_q \\(if set\\) must be the same type as notch"),
    ("notch = 100.0; notch_q = 0.0;", "invalid value for notch_q"),
    ("ctcss = 100;", "ctcss should be an float"),
    ("ampfactor = -1.0;", "must not be negative"),
    ("ampfactor = 2;", "invalid parameter type: devices.\\[0\\].channels.\\[0\\].ampfactor"),
    ("afc = -1;", "invalid parameter type"),
    ("tau = 1.5;", "invalid parameter type"),
    ('disable = "no";', "invalid parameter type"),
])
def test_channel_errors_are_the_references(body, message):
    with pytest.raises(host.ConfigError, match=message) as ei:
        one_channel(body)
    assert ei.value.code == host.ERR_CONFIG


def test_missing_and_malformed_structure():
    with pytest.raises(host.ConfigError, match="mandatory parameter missing: devices"):
        host.parse_text("fft_size = 512;")
    with pytest.raises(host.ConfigError, match="mandatory parameter missing: devices.\\[0\\].centerfreq"):
        host.parse_text('devices: ({ type = "rtlsdr"; channels: ({ freq = 1.0; %s }); });' % OUT)
    with pytest.raises(host.ConfigError, match="mandatory parameter missing: devices.\\[0\\].channels.\\[0\\].freq"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ %s }); });' % OUT)
    with pytest.raises(host.ConfigError, match="mandatory parameter missing: devices.\\[0\\].channels.\\[0\\].outputs"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; }); });')
    with pytest.raises(host.ConfigError, match="no outputs defined"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; outputs: (); }); });')
    with pytest.raises(host.ConfigError, match="no outputs defined"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; outputs: ({ type = "file"; disable = true; }); }); });')
    with pytest.raises(host.ConfigError, match="unknown output type"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; outputs: ({ type = "tape"; }); }); });')
    with pytest.raises(host.ConfigError, match="unknown mixer"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; outputs: ({ type = "mixer"; name = "m1"; }); }); });')
    with pytest.raises(host.ConfigError, match="no devices defined"):
        host.parse_text("devices: ();")
    with pytest.raises(host.ConfigError, match="no devices defined"):
        host.parse_text('devices: ({ disable = true; });')
    with pytest.raises(host.ConfigError, match="no channels configured"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: (); });')
    with pytest.raises(host.ConfigError, match="no channels enabled"):
        host.parse_text('devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; disable = true; %s }); });' % OUT)
    with pytest.raises(host.ConfigError, match="unsupported device type"):
        host.parse_text('devices: ({ type = "hackrf"; centerfreq = 1.0; channels: ({ freq = 1.0; %s }); });' % OUT)
    with pytest.raises(host.ConfigError, match="invalid fft_size value"):
        host.parse_text("fft_size = 500;" + BASIC.replace("fft_size = 512;", ""))
    with pytest.raises(host.ConfigError, match="sample_rate must be greater than 8000"):
        host.parse_text('devices: ({ type = "rtlsdr"; sample_rate = 4000; centerfreq = 1.0; channels: ({ freq = 1.0; %s }); });' % OUT, 8000)
    with pytest.raises(host.ConfigError, match="invalid mode"):
        host.parse_text('devices: ({ type = "rtlsdr"; mode = "sweep"; centerfreq = 1.0; channels: ({ freq = 1.0; %s }); });' % OUT)
    # a mixer output naming a defined mixer is fine
    ok = 'mixers: { m1: { %s } }; devices: ({ type = "rtlsdr"; centerfreq = 1.0; channels: ({ freq = 1.0; outputs: ({ type = "mixer"; name = "m1"; }); }); });' % OUT
    assert len(host.parse_text(ok).cfg.devices[0].channels) == 1


MIXERS = """
mixers: {
  tower: { outputs: ( { type = "icecast"; server = "x"; port = 8000; mountpoint = "m"; username = "u"; password = "p"; } ); },
  off:   { disable = true; %(o)s },
  wide:  { highpass = 200; lowpass = 3000; %(o)s }
};
devices: (
  { type = "rtlsdr"; centerfreq = 120.0; channels: (
      { freq = 119.5; outputs: ( { type = "mixer"; name = "tower"; }, { type = "mixer"; name = "wide"; balance = -0.5; ampfactor = 2.0; } ); },
      { freq = 119.7; squelch_snr_threshold = -1; outputs: ( { type = "mixer"; name = "tower"; } ); },
      { freq = 119.9; outputs: ( { type = "mixer"; name = "tower"; disable = true; }, { type = "mixer"; name = "wide"; balance = 1.0; }, { type = "file"; directory = "/tmp"; filename_template = "x"; } ); } ); },
  { disable = true; type = "rtlsdr"; centerfreq = 130.0; channels: ( { freq = 130.1; outputs: ( { type = "mixer"; name = "tower"; } ); } ); },
  { type = "rtlsdr"; centerfreq = 125.0; channels: ( { freq = 125.1; outputs: ( { type = "mixer"; name = "tower"; ampfactor = 0.5; } ); } ); }
);
""" % {"o": OUT}


def test_mixers_connect_in_the_references_order():
    """parse_mixers runs first (config.cpp:838-889); every enabled channel output of type "mixer" then connects as the next
    input of the mixer it names (config.cpp:173-194, mixer.cpp:55-93).  Disabled mixers do not exist for getmixerbyname."""
    c = host.parse_text(MIXERS)
    mx = c.cfg.mixers
    assert [m.name for m in mx] == ["tower", "wide"]
    # the dropped channel (squelch_snr_threshold = -1) never reaches its outputs; device indices count enabled devices
    assert [(i.device, i.channel, i.ampfactor, i.balance) for i in mx[0].inputs] == [(0, 0, 1.0, 0.0), (1, 0, 0.5, 0.0)]
    assert [(i.device, i.channel, i.ampfactor, i.balance) for i in mx[1].inputs] == [(0, 0, 2.0, -0.5), (0, 1, 1.0, 1.0)]
    assert not mx[0].stereo and mx[1].stereo
    for bad, msg in [
        (MIXERS.replace('name = "wide"; balance = 1.0', 'name = "wide"; balance = 1.5'), "balance out of allowed range"),
        (MIXERS.replace('name = "wide"; balance = 1.0', 'name = "off"'), 'unknown mixer "off"'),
        (MIXERS.replace('ampfactor = 0.5', 'ampfactor = 1'), "invalid parameter type"),
        (MIXERS.replace("highpass = 200; lowpass = 3000;", "highpass = 200; lowpass = 100;"), r"mixers.\[2\]: lowpass \(100\) must be greater"),
        (MIXERS.replace('tower: { outputs: ( { type = "icecast";', 'tower: { outputs: ( { type = "rawfile";'), "rawfile output is not allowed for mixers"),
        (MIXERS.replace('tower: { outputs: ( { type = "icecast";', 'tower: { outputs: ( { type = "mixer"; name = "wide";'), "mixer output is not allowed for mixers"),
        (MIXERS.replace('tower: { outputs: ( { type = "icecast";', 'tower: { outputs: ( { disable = true; type = "icecast";'), r"mixers.\[0\]: no outputs defined"),
    ]:
        with pytest.raises(host.ConfigError, match=msg):
            host.parse_text(bad)


SCAN = """
fft_size = 1024;
devices: ({ type = "rtlsdr"; sample_rate = 2.4; mode = "scan";
  channels: ({
    freqs = ( 162.4, 162550000, "156.8M" );
    labels = ( "a", "b", "c" );
    modulations = ( "nfm", "am", "nfm" );
    squelch_threshold = ( -40, 0, -55 );
    squelch_snr_threshold = ( 6.0, -1, 3 );
    notch = ( 100.0, 0.0, 250.0 ); notch_q = ( 0.0, 5.0, 4.0 );
    ctcss = ( 0.0, 0.0, 88.5 );
    bandwidth = ( 12500, 0, "8k" );
    ampfactor = ( 1.0, 2.0, 0.5 );
    afc = 3; tau = 300;
    %(o)s }); });
""" % {"o": OUT}


def test_scan_mode_frequency_lists():
    """R_SCAN (config.cpp:364-433): one channel, per-frequency lists, centre frequency 20 bins above the first frequency."""
    c = host.parse_text(SCAN)
    assert c.is_scan(0) and c.cfg.wave_rate == 16000
    d = c.cfg.devices[0]
    assert d.centerfreq == int(int(162.4 * 1e6) + 20 * float(2400000 // 1024))
    ch = d.channels[0]
    assert (ch.afc, ch.tau, len(ch.freqs)) == (3, 300, 3)
    f = ch.freqs
    assert [x.freq for x in f] == [int(162.4 * 1e6), 162550000, 156800000]
    assert [x.modulation for x in f] == ["nfm", "am", "nfm"]
    assert [x.squelch_threshold for x in f] == [-40, 0, -55]
    assert [x.squelch_snr_threshold for x in f] == [6.0, -1.0, 3.0]  # -1 in a list keeps the default for that frequency
    assert [(x.notch, x.notch_q) for x in f] == [(100.0, 10.0), (0.0, 0.0), (250.0, 4.0)]  # q 0 = default 10; notch 0 = off
    assert [x.ctcss for x in f] == [0.0, 0.0, 88.5] and [x.bandwidth for x in f] == [12500, 0, 8000] and [x.ampfactor for x in f] == [1.0, 2.0, 0.5]
    assert (ch.freq, ch.modulation, ch.bandwidth, ch.notch) == (f[0].freq, "nfm", 12500, 100.0)  # the channel's own fields repeat freqlist[0]
    # scalars apply to every frequency
    c2 = host.parse_text(SCAN.replace('modulations = ( "nfm", "am", "nfm" );', 'modulation = "nfm";').replace("ampfactor = ( 1.0, 2.0, 0.5 );", "ampfactor = 3.0;"))
    assert [x.modulation for x in c2.cfg.devices[0].channels[0].freqs] == ["nfm"] * 3 and [x.ampfactor for x in c2.cfg.devices[0].channels[0].freqs] == [3.0] * 3
    for bad, msg in [
        (SCAN.replace("freqs = ( 162.4, 162550000, \"156.8M\" );", "freqs = ( );"), "freqs should be a list with at least one element"),
        (SCAN.replace('labels = ( "a", "b", "c" );', 'labels = ( "a" );'), "labels should be a list with at least 3 elements"),
        (SCAN.replace("squelch_threshold = ( -40, 0, -55 );", "squelch_threshold = ( -40 );"), "squelch_threshold should be an int or a list of ints with at least 3 elements"),
        (SCAN.replace("ctcss = ( 0.0, 0.0, 88.5 );", "ctcss = ( 0.0 );"), "ctcss should be an float or a list of floats with at least 3 elements"),
        (SCAN.replace('modulations = ( "nfm", "am", "nfm" );', 'modulations = ( "nfm", "am", "nfm" ); modulation = "am";'), "can't set both modulation and modulations"),
        (SCAN.replace('modulations = ( "nfm", "am", "nfm" );', 'modulations = ( "nfm", "usb", "nfm" );'), r"modulations.\[1\]: unknown modulation"),
        (SCAN.replace("notch_q = ( 0.0, 5.0, 4.0 );", "notch_q = ( 0.0, -5.0, 4.0 );"), r"freq.\[1\]: invalid value for notch_q"),
        (SCAN.replace("%s }); });" % OUT, "%s }, { freqs = ( 1.0 ); %s }); });" % (OUT, OUT)), "only one channel is allowed in scan mode"),
        (SCAN.replace("freqs = ", "freq = 1.0; nofreqs = "), r"mandatory parameter missing: devices.\[0\].channels.\[0\].freqs"),
    ]:
        with pytest.raises(host.ConfigError, match=msg):
            host.parse_text(bad)


def test_scan_controller_follows_the_references_thread():
    """controller_thread (boondock_airband.cpp:101-139): polled every 200 ms; after 10 consecutive polls without signal it moves
    to the next frequency at every further poll, a poll with signal resets the count (and tags the frequency once)."""
    L = host.load_library()
    st = (C.c_int32 * 4)(0, 0, -1, 3)  # i, consecutive_squelch_off, last_frequency, freq_count
    L.ba_scan_controller_poll.argtypes = [C.POINTER(C.c_int32), C.c_int, C.POINTER(C.c_int)]
    seq, tags = [], []
    polls = [0] * 13 + [1, 1] + [0] * 12 + [1]
    for has_signal in polls:
        tag = C.c_int(-1)
        seq.append(L.ba_scan_controller_poll(st, has_signal, C.byref(tag)))
        tags.append(tag.value)
    # model of the loop
    i = off = 0
    last = -1
    want, want_tags = [], []
    for has_signal in polls:
        tag = -1
        if not has_signal:
            if off < 10:
                off += 1
            else:
                i = (i + 1) % 3
        else:
            if off == 10 and i != last:
                tag = last = i
            off = 0
        want.append(i)
        want_tags.append(tag)
    assert seq == want and tags == want_tags
    assert seq[9] == 0 and seq[10] == 1 and seq[12] == 0 and seq[13] == 0 and tags[13] == 0 and tags[14] == -1
    one = (C.c_int32 * 4)(0, 0, -1, 1)  # freq_count < 2: the thread returns at once (:108-109)
    assert [L.ba_scan_controller_poll(one, 0, None) for _ in range(15)] == [0] * 15


def test_missing_type_falls_back_to_rtlsdr_with_the_warning():
    c = host.parse_text('devices: ({ centerfreq = 1.0; channels: ({ freq = 1.0; %s }); });' % OUT)
    assert c.cfg.devices[0].sample_rate == 2560000
    assert any('assuming device type "rtlsdr"' in w for w in c.warnings)


def test_the_two_silent_channel_drops():
    """`continue` at config.cpp:504-506 and :612-614 leaves the channel loop: the entry vanishes, the slot is reused, and
    the slot's needs_raw_iq (set at :592 before the second `continue`) sticks to the entry that takes the slot."""
    text = ('devices: ({ type = "rtlsdr"; centerfreq = 120.0; channels: ('
            '{ freq = 120.1; squelch_snr_threshold = -1; %(o)s }, { freq = 120.2; %(o)s },'
            '{ freq = 120.3; bandwidth = 0; %(o)s }, { freq = 120.4; %(o)s }, { freq = 120.5; %(o)s },'
            '{ freq = 120.6; squelch_snr_threshold = -1.0; %(o)s }, { freq = 120.7; squelch_snr_threshold = (-1.0); %(o)s } ); });' % {"o": OUT})
    c = host.parse_text(text, 16000)
    ch = c.cfg.devices[0].channels
    assert [x.freq for x in ch] == [int(f * 1e6) for f in (120.2, 120.4, 120.5, 120.7)]
    assert [c.source_index(0, k) for k in range(4)] == [1, 3, 4, 6]
    assert [x.bandwidth for x in ch] == [0, -1, 0, 0]  # -1 = raw-IQ path on, no filter
    assert ch[3].squelch_snr_threshold == -1.0  # in list form -1 keeps the default and the channel
    assert sum("dropped without a message" in w for w in c.warnings) == 3


def test_warnings_of_the_reference():
    c = one_channel("squelch = 10; squelch_threshold = -30; squelch_snr_threshold = 5.0; notch = -5.0; ctcss = -1.0; bandwidth = -3;")
    w = "\n".join(c.warnings)
    assert "'squelch' no longer supported" in w and "may conflict" in w
    assert "notch value '-5' invalid, ignoring" in w and "ctcss value '-1' invalid, ignoring" in w and "bandwidth value '-3' invalid, ignoring" in w
    ch = c.cfg.devices[0].channels[0]
    assert (ch.notch, ch.ctcss, ch.bandwidth, ch.squelch_threshold, ch.squelch_snr_threshold) == (0.0, 0.0, -1, -30, 5.0)


def test_list_forms_take_the_single_frequency():
    c = one_channel("squelch_threshold = (-35); squelch_snr_threshold = (7); notch = (250.0); notch_q = (0.0); ctcss = (88.5); bandwidth = (8000); ampfactor = (1.5);")
    ch = c.cfg.devices[0].channels[0]
    assert (ch.squelch_threshold, ch.squelch_snr_threshold, ch.notch, ch.notch_q, ch.ctcss, ch.bandwidth, ch.ampfactor) == (-35, 7.0, 250.0, 10.0, 88.5, 8000, 1.5)


def test_grammar_subset(tmp_path):
    inc = tmp_path / "chan.inc"
    inc.write_text('freq = 0x7270E00; /* 120 MHz in hex */ label = "a" "b\\n\\x41\\"";\n' + OUT)
    main = tmp_path / "main.conf"
    main.write_text('''
/* block
   comment */
fft_size : 2048   # colon and no semicolon
big = 5000000000; wide = 7L; arr = [ 1, 2, 3 ]; farr = [ 1.5, 2e3, .5 ]; empty = ( ); flag = TRUE;
devices = ( { type = "file"; filepath = "/dev/null"; speedup_factor = 2.5; sample_rate = 2.56; sample_format = "f32";
              centerfreq = 120e0,
              channels = ( { @include "chan.inc" } ) } )
''')
    c = host.parse_file(str(main))
    d = c.cfg.devices[0]
    assert c.cfg.fft_size == 2048 and d.centerfreq == 120000000 and d.channels[0].freq == 0x7270E00
    assert (d.sample_format, d.bytes_per_sample, d.fullscale) == ("f32", 4, 1.0)
    assert c.setting(0, "filepath") == "/dev/null" and float(c.setting(0, "speedup_factor")) == 2.5
    for bad, msg in [("a = ;", "line 1"), ("a = 1\nb = [1, \"x\"];", "line 2.*mismatched"), ('a = "unterminated', "unterminated string"),
                     ("a = 1; a = 2;", "duplicate setting"), ("a = { b = 1;", "unexpected end"), ("a = 1; }", "unmatched"), ("a = 12abc;", "syntax error"),
                     ("/* x", "unterminated comment"), ('@include "/nonexistent/file"', "Cannot read configuration file")]:
        with pytest.raises(host.ConfigError, match=msg) as ei:
            host.parse_text(bad)
        assert ei.value.code in (host.ERR_SYNTAX, host.ERR_IO)
    with pytest.raises(host.ConfigError, match="Cannot read configuration file"):
        host.parse_file(str(tmp_path / "missing.conf"))


def test_file_driver_checks():
    base = 'devices: ({ type = "file"; %s centerfreq = 120.0; channels: ({ freq = 120.1; %s }); });'
    with pytest.raises(host.ConfigError, match="no 'filepath' given"):
        host.parse_text(base % ("sample_rate = 2.56;", OUT))
    with pytest.raises(host.ConfigError, match="'speedup_factor' must be >= 0.0"):
        host.parse_text(base % ('filepath = "x"; sample_rate = 2.56; speedup_factor = 0;', OUT))
    with pytest.raises(host.ConfigError, match="'speedup_factor' must be a float or int"):
        host.parse_text(base % ('filepath = "x"; sample_rate = 2.56; speedup_factor = "2";', OUT))
    with pytest.raises(host.ConfigError, match="sample_rate must be greater than"):  # file_input_new leaves sample_rate 0 (config.cpp:793)
        host.parse_text(base % ('filepath = "x";', OUT))
    with pytest.raises(host.ConfigError, match="sample_format must be one of"):
        host.parse_text(base % ('filepath = "x"; sample_rate = 2.56; sample_format = "s24";', OUT))
    with pytest.raises(host.ConfigError, match='set "sample_format"'):
        host.parse_text('devices: ({ type = "soapysdr"; sample_rate = 2.56; centerfreq = 120.0; channels: ({ freq = 120.1; %s }); });' % OUT)


@pytest.mark.skipif(not os.path.isdir(REF_CONFIGS), reason="the reference tree is not mounted")
def test_the_references_own_configuration_files():
    """Every multichannel example of the reference loads unchanged; derived bins follow config.cpp:669-670."""
    seen = scans = 0
    for name in sorted(os.listdir(REF_CONFIGS)):
        path = os.path.join(REF_CONFIGS, name)
        text = open(path).read()
        c = host.parse_file(path)
        for k, d in enumerate(c.cfg.devices):
            if c.is_scan(k):
                f0 = d.channels[0].freqs[0].freq
                assert len(d.channels) == 1 and d.centerfreq == int(f0 + 20 * float(d.sample_rate // c.cfg.fft_size))  # config.cpp:431
                scans += 1
        n_entries = len(re.findall(r"^\s*freqs?\s*=", text, re.M))
        assert sum(len(d.channels) for d in c.cfg.devices) == n_entries, name
        assert sum(len(m.inputs) for m in c.cfg.mixers) == len(re.findall(r'type\s*=\s*"mixer"', text)), name
        for d in c.cfg.devices:
            for ch in d.channels:
                b = int(math.ceil((ch.freq + d.sample_rate - d.centerfreq) / float(d.sample_rate // c.cfg.fft_size) - 1.0)) % c.cfg.fft_size
                assert 0 <= b < c.cfg.fft_size
        seen += 1
    assert seen >= 6 and scans >= 2
    sc = host.parse_file(os.path.join(REF_CONFIGS, "basic_scanning.conf")).cfg.devices[0].channels[0]
    assert [f.freq for f in sc.freqs] == [int(f * 1e6) for f in (118.15, 124.7, 132.1)]
    noaa = host.parse_file(os.path.join(REF_CONFIGS, "noaa.conf")).cfg
    assert noaa.wave_rate == 16000 and noaa.fft_size == 1024 and noaa.devices[0].sample_rate == int(2.40 * 1e6)
    assert all(ch.modulation == "nfm" and ch.bandwidth == 5000 and ch.squelch_snr_threshold == 0.0 and ch.ampfactor == 2.0 for ch in noaa.devices[0].channels)


def test_parsed_model_builds_the_same_descriptor_as_the_hand_written_one(oracle_built):
    """A file saying what configs.cfg1() says gives the oracle the same bins and constants."""
    from boondock_airband_b200 import configs
    from oracle.ba_oracle import Oracle

    want = configs.cfg1()
    text = 'fft_size = 512; devices: ({ type = "rtlsdr"; centerfreq = 120000000; sample_rate = 2560000; channels: (%s); });' % ",".join(
        "{ freq = %d; %s }" % (ch.freq, OUT) for ch in want.devices[0].channels)
    got = host.parse_text(text, 8000).cfg
    a, b = Oracle(want), Oracle(got)
    for ch in range(len(want.devices[0].channels)):
        assert a.channel_info(0, ch).as_dict() == b.channel_info(0, ch).as_dict()


# ------------------------------------------------------------------------------------------------ file input

class PyRing:
    """An input_t ring kept in Python (input-common.h:39-57) behind the ba_ring_sink callbacks."""
    SPACE = C.CFUNCTYPE(C.c_size_t, C.c_void_p)
    APPEND = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)

    def __init__(self, size):
        self.size, self.taken, self.calls, self.fail_after = size, 0, [], None
        self.data = bytearray()
        self._space = self.SPACE(lambda ctx: self.size - (len(self.data) - self.taken) - 1)
        self._append = self.APPEND(self.append)
        self.sink = host.RingSink(None, C.cast(self._space, C.c_void_p), C.cast(self._append, C.c_void_p))

    def append(self, ctx, ptr, n):
        if self.fail_after is not None and len(self.calls) >= self.fail_after:
            return -6
        assert n <= self.size - (len(self.data) - self.taken) - 1
        self.calls.append(n)
        self.data += C.string_at(ptr, n)
        return 0


def open_input(path, ring, **kw):
    L = host.load_library()
    d = dict(sample_format=abi.SFMT["u8"], sample_rate=0, speedup_factor=0.0, chunk_bytes=0, ring_bytes=ring.size, loop=0)
    d.update(kw)
    desc = host.FileInputDesc(str(path).encode(), d["sample_format"], d["sample_rate"], d["speedup_factor"], d["chunk_bytes"], d["ring_bytes"], d["loop"])
    h = C.c_void_p()
    rc = L.ba_file_input_open(C.byref(desc), C.byref(ring.sink), C.byref(h))
    return L, rc, h


def wait_for(cond, timeout=10.0):
    t0 = time.time()
    while not cond():
        if time.time() - t0 > timeout:
            return False
        time.sleep(0.002)
    return True


def test_file_input_replays_the_file_in_order(tmp_path):
    rng = np.random.default_rng(7)
    payload = rng.integers(0, 256, 100_003, dtype=np.uint8).tobytes()  # odd length: the last byte is half a sample
    p = tmp_path / "iq.u8"
    p.write_bytes(payload)
    ring = PyRing(20_000)
    L, rc, h = open_input(p, ring)
    assert rc == 0 and L.ba_file_input_state(h) == host.INPUT_INITIALIZED
    assert L.ba_file_input_start(h) == 0
    consumed = 0

    def drain():
        nonlocal consumed
        ring.taken = len(ring.data)  # the demodulator takes everything
        consumed = ring.taken
        return L.ba_file_input_state(h) == host.INPUT_FAILED  # end of file, as input-file.cpp:107-111

    assert wait_for(drain)
    assert bytes(ring.data) == payload[:100_002] and L.ba_file_input_bytes(h) == 100_002
    # chunk = buf_size/2 - 1 (input-file.cpp:96), rounded down to whole complex samples
    assert max(ring.calls) == 9998 and all(n % 2 == 0 for n in ring.calls)
    assert L.ba_file_input_start(h) == -7
    assert L.ba_file_input_stop(h) == 0


def test_file_input_waits_for_space_and_stops(tmp_path):
    p = tmp_path / "iq.s16"
    p.write_bytes(bytes(range(256)) * 400)
    ring = PyRing(10_000)
    L, rc, h = open_input(p, ring, sample_format=abi.SFMT["s16"], chunk_bytes=4098, loop=1)
    assert rc == 0 and L.ba_file_input_start(h) == 0
    assert wait_for(lambda: len(ring.calls) == 2)
    time.sleep(0.05)
    assert len(ring.calls) == 2 and ring.calls == [4096, 4096]  # 4098 rounded to whole 4-byte samples; the third read waits
    ring.taken = len(ring.data)
    assert wait_for(lambda: len(ring.calls) >= 4)
    assert L.ba_file_input_state(h) == host.INPUT_RUNNING
    assert L.ba_file_input_stop(h) == 0  # joins the reader
    n = len(ring.data)
    assert bytes(ring.data) == (bytes(range(256)) * (n // 256 + 1))[:n]  # loop=1 rewinds seamlessly (102400 is a multiple of 4096)


def test_file_input_pacing_follows_speedup_factor(tmp_path):
    """time_per_byte_ms = 1000 / (Fs * bytes_per_sample * 2 * speedup) (input-file.cpp:99): 100 kB of u8 IQ at 1 Msps x2 is 25 ms."""
    p = tmp_path / "iq.u8"
    p.write_bytes(bytes(200_000))
    ring = PyRing(1 << 20)
    L, rc, h = open_input(p, ring, sample_rate=1_000_000, speedup_factor=2.0, chunk_bytes=20_000)
    t0 = time.time()
    assert rc == 0 and L.ba_file_input_start(h) == 0
    assert wait_for(lambda: L.ba_file_input_state(h) == host.INPUT_FAILED)
    dt = time.time() - t0
    assert 0.04 <= dt <= 0.5, dt  # 10 reads x 5 ms of sleep each = 50 ms (int ms arithmetic shaves a little)
    assert L.ba_file_input_stop(h) == 0 and len(ring.data) == 200_000


def test_file_input_errors(tmp_path):
    ring = PyRing(1000)
    L, rc, h = open_input(tmp_path / "missing", ring)
    assert rc == host.ERR_IO and b"failed to open" in L.ba_host_last_error()
    p = tmp_path / "x"
    p.write_bytes(bytes(5000))
    assert open_input(p, ring, sample_format=9)[1] == -4
    assert open_input(p, ring, speedup_factor=-1.0)[1] == host.ERR_CONFIG
    assert open_input(p, ring, speedup_factor=1.0)[1] == -4  # paced replay needs the rate
    ring.fail_after = 1
    L, rc, h = open_input(p, ring, chunk_bytes=100)
    assert rc == 0 and L.ba_file_input_start(h) == 0
    assert wait_for(lambda: L.ba_file_input_state(h) == host.INPUT_FAILED)  # a refused append fails the input
    assert len(ring.data) == 100 and L.ba_file_input_stop(h) == 0


def test_handoff_keeps_order_and_applies_back_pressure():
    """Row f-4: the waveavail/Signal hand-off (boondock_airband.cpp:673-679,728; output.cpp:899-961) with N slots."""
    import threading
    L = host.load_library()
    h = C.c_void_p()
    assert L.ba_handoff_create(0, 16, C.byref(h)) == -4
    assert L.ba_handoff_create(3, 4000, C.byref(h)) == 0
    n_batches, got, slow = 40, [], 0.002

    def output_thread():
        slot, tag = C.c_void_p(), C.c_uint64()
        while True:
            rc = L.ba_handoff_take(h, -1, C.byref(slot), C.byref(tag))
            if rc == host.HANDOFF_CLOSED:
                return
            assert rc == 0 and slot.value % 64 == 0
            a = np.ctypeslib.as_array(C.cast(slot, C.POINTER(C.c_float)), shape=(1000,))
            got.append((tag.value, float(a[0]), float(a[-1])))
            time.sleep(slow)  # a slow encoder
            assert L.ba_handoff_release(h, slot) == 0

    t = threading.Thread(target=output_thread)
    t.start()
    t0 = time.time()
    for k in range(n_batches):  # the demodulator: far faster than the consumer
        slot = C.c_void_p()
        assert L.ba_handoff_acquire(h, -1, C.byref(slot)) == 0
        a = np.ctypeslib.as_array(C.cast(slot, C.POINTER(C.c_float)), shape=(1000,))
        a[:] = k
        assert L.ba_handoff_publish(h, slot, 1000 + k) == 0
    produced_in = time.time() - t0
    L.ba_handoff_close(h)  # do_exit: the consumer drains what is queued, then leaves
    t.join(10)
    assert not t.is_alive()
    assert got == [(1000 + k, float(k), float(k)) for k in range(n_batches)]  # nothing lost, nothing reordered
    assert produced_in >= (n_batches - 4) * slow  # the producer was held back to the consumer's pace
    assert L.ba_handoff_overruns(h) == 0
    slot = C.c_void_p()
    assert L.ba_handoff_acquire(h, -1, C.byref(slot)) == host.HANDOFF_CLOSED
    L.ba_handoff_destroy(h)


def test_handoff_polling_counts_overruns_like_the_reference():
    L = host.load_library()
    h = C.c_void_p()
    assert L.ba_handoff_create(2, 64, C.byref(h)) == 0
    s = [C.c_void_p() for _ in range(3)]
    assert L.ba_handoff_acquire(h, 0, C.byref(s[0])) == 0 and L.ba_handoff_acquire(h, 0, C.byref(s[1])) == 0
    assert L.ba_handoff_acquire(h, 0, C.byref(s[2])) == host.HANDOFF_TIMEOUT and L.ba_handoff_overruns(h) == 1  # output_overrun_count++
    assert L.ba_handoff_acquire(h, 5, C.byref(s[2])) == host.HANDOFF_TIMEOUT and L.ba_handoff_overruns(h) == 2
    taken, tag = C.c_void_p(), C.c_uint64()
    assert L.ba_handoff_take(h, 0, C.byref(taken), C.byref(tag)) == host.HANDOFF_TIMEOUT  # nothing published yet
    assert L.ba_handoff_release(h, s[0]) == -7 and L.ba_handoff_publish(h, C.c_void_p(s[0].value + 8), 0) == -4
    assert L.ba_handoff_publish(h, s[1], 7) == 0 and L.ba_handoff_publish(h, s[1], 7) == -7
    assert L.ba_handoff_take(h, 0, C.byref(taken), C.byref(tag)) == 0 and taken.value == s[1].value and tag.value == 7
    assert L.ba_handoff_release(h, taken) == 0
    assert L.ba_handoff_acquire(h, 0, C.byref(s[2])) == 0 and s[2].value == s[1].value
    L.ba_handoff_destroy(h)


def test_host_header_binding_and_exports_agree(tmp_path):
    names = sorted(set(re.findall(r"^BA_HOST_API\s+[\w\s\*]+?\b(ba_\w+)\s*\(", open(HEADER).read(), re.M)))
    assert names == sorted(host.SYMBOLS)
    out = subprocess.check_output(["nm", "-D", "--defined-only", host.DEFAULT_LIB], text=True)
    assert set(re.findall(r"\bT (ba_\w+)", out)) == set(names)
    assert "cuda" not in subprocess.check_output(["ldd", host.DEFAULT_LIB], text=True)  # loads on a machine without CUDA
    src = tmp_path / "ba_host_c99.c"
    src.write_text('#include "ba_host.h"\nint main(void){return BA_OK;}\n')
    subprocess.check_call(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", "-o", str(tmp_path / "ba_host_c99.o"), str(src)])
