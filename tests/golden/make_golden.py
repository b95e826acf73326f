#!/usr/bin/env python
"""Generates the golden fixtures under tests/golden/ from the REFERENCE-BUILT oracle (oracle/_ref/libba_oracle_ref.so:
the reference's own squelch.cpp, ctcss.cpp and filters.cpp compiled unmodified from /root/reference/src and driven by
the restated demodulate() loop).  Runs only where /root/reference is mounted; the .npz files it writes are committed
so that the restated oracle and the CUDA path can be pinned anywhere.

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from boondock_airband_b200 import abi, synth  # noqa: E402
from oracle import ba_oracle  # noqa: E402
from oracle.ba_oracle import Oracle, SquelchProbe  # noqa: E402
import golden_cases  # noqa: E402


def pipeline_case(name):
    cfg, iq = golden_cases.build(name)
    o = Oracle(cfg, ref=True)
    o.feed(0, iq)
    nch = len(cfg.devices[0].channels)
    out = dict(iq=iq, frames=np.int64(o.frames(0)), batches=np.int64(o.batches(0)))
    out["waveout"] = np.stack([o.waveout(0, c) for c in range(nch)])
    out["trace"] = np.stack([o.trace(0, c) for c in range(nch)])
    out["picks"] = np.stack([o.picks(0, c) for c in range(nch)])
    info = [o.channel_info(0, c) for c in range(nch)]
    out["bins"] = np.array([i.bin for i in info], np.uint32)
    out["dm_dphi"] = np.array([i.dm_dphi for i in info], np.uint32)
    out["info_raw"] = np.stack([np.frombuffer(bytes(i), np.uint8) for i in info])
    st = []
    for c in range(nch):
        st.append(np.array([[s.axcindicate, s.bin, s.open_count, s.flappy_count, s.ctcss_count, s.no_ctcss_count, s.active_counter] for s in o.status(0, c)], np.int64))
    out["status_int"] = np.stack(st)
    lv = []
    for c in range(nch):
        lv.append(np.array([[s.signal_level, s.noise_level, s.squelch_level] for s in o.status(0, c)], np.float32))
    out["status_levels"] = np.stack(lv)
    iqc = [c for c in range(nch) if cfg.devices[0].channels[c].has_iq_outputs]
    if iqc:
        out["iq_out"] = np.stack([o.iq_out(0, c) for c in iqc])
        out["iq_channels"] = np.array(iqc)
    np.savez_compressed(os.path.join(HERE, name + "_iq.npz"), iq=out.pop("iq"))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "frames", out["frames"], "batches", out["batches"], "open samples", int(((out["trace"] & abi.TRACE_OPEN) != 0).sum()))


def dsp_case():
    """Bare DSP objects of the reference on seeded stimuli: squelch state/level traces, CTCSS decisions, filters."""
    rng = np.random.default_rng(0xB00D)
    out = {}
    # squelch: noise, signal, dead spot, flapping bursts, weak signal (low-signal abort), with and without post-filter samples
    raw = np.concatenate([np.full(3000, 0.05), np.full(1500, 0.75), np.full(50, 0.05), np.full(800, 0.75), np.full(600, 0.05)]
                         + [np.concatenate([np.full(260, 0.75), np.full(300, 0.05)]) for _ in range(5)]
                         + [np.full(400, 0.75), np.tile(np.array([0.75, 0.01, 0.01, 0.01], np.float32), 150), np.full(500, 0.05)]).astype(np.float32)
    raw = (raw * (1.0 + 0.05 * rng.standard_normal(raw.size))).astype(np.float32)
    filt = (raw * np.where(rng.random(raw.size) < 0.1, 0.2, 0.95)).astype(np.float32)
    audio = (0.2 * np.sin(2 * np.pi * 100.0 * np.arange(raw.size) / 8000.0)).astype(np.float32)
    out["sq_raw"], out["sq_filtered"], out["sq_audio"] = raw, filt, audio
    for tag, kw in (("plain", {}), ("filtered", dict(filtered=filt)), ("ctcss", dict(audio=audio, ctcss=100.0)), ("manual", dict(level=0.3))):
        p = SquelchProbe(ref=True)
        if "ctcss" in kw:
            p.set_ctcss(kw["ctcss"], 8000.0)
        if "level" in kw:
            p.set_level(kw["level"])
        st, lv = p.run(raw, kw.get("filtered"), kw.get("audio"), want_levels=True)
        q = p.query()
        out["sq_states_" + tag], out["sq_levels_" + tag] = st, lv
        out["sq_counts_" + tag] = np.array([q["open_count"], q["flappy_count"], q["ctcss_count"], q["no_ctcss_count"]], np.int64)
    # CTCSS: each standard tone against a detector for every standard tone, slow window at 8 kHz, seeded noise
    tones = np.array([67.0, 69.3, 71.9, 74.4, 77.0, 79.7, 82.5, 85.4, 88.5, 91.5, 94.8, 97.4, 100.0, 103.5, 107.2, 110.9, 114.8, 118.8, 123.0, 127.3, 131.8, 136.5,
                      141.3, 146.2, 150.0, 151.4, 156.7, 159.8, 162.2, 165.5, 167.9, 171.3, 173.8, 177.3, 179.9, 183.5, 186.2, 189.9, 192.8, 196.6, 199.5, 203.5,
                      206.5, 210.7, 218.1, 225.7, 229.1, 233.6, 241.8, 250.3, 254.1], np.float32)
    n = 3200
    t = np.arange(1, n + 1)
    sig = np.stack([(0.2 * np.sin(2 * np.pi * t * float(f) / 8000.0) + 0.2 * 0.1 * rng.standard_normal(n)).astype(np.float32) for f in tones])
    dec = np.zeros((tones.size, tones.size), np.uint8)
    for i in range(tones.size):
        for j in range(tones.size):
            tone, enough = ba_oracle.ctcss_run(float(tones[j]), 8000.0, 3200, sig[i], ref=True)
            assert enough
            dec[i, j] = tone
    out["ctcss_tones"], out["ctcss_signals"], out["ctcss_decisions"] = tones, sig, dec
    # filters
    x = (0.5 * rng.standard_normal(2000)).astype(np.float32)
    y, _ = ba_oracle.notch_run(100.0, 16000.0, 10.0, x, ref=True)
    out["notch_in"], out["notch_out"] = x, y
    z = (rng.standard_normal(2000) + 1j * rng.standard_normal(2000)).astype(np.complex64)
    out["lp_in"], out["lp_out"] = z, ba_oracle.lowpass_run(6250.0, 16000.0, z, ref=True).astype(np.complex64)
    np.savez_compressed(os.path.join(HERE, "dsp_objects.npz"), **out)
    print("dsp_objects written; ctcss diagonal hits", int(np.trace(dec)), "off-diagonal hits", int(dec.sum() - np.trace(dec)))


if __name__ == "__main__":
    if not ba_oracle.have_ref():
        ba_oracle.build(ref=True)
    assert ba_oracle.load(ref=True).ba_oracle_is_reference_build() == 1
    for name in golden_cases.NAMES:
        pipeline_case(name)
    dsp_case()
