"""The configurations behind the committed golden fixtures (tests/golden/*.npz).  Sample rates are kept low so that the
input IQ itself fits in the fixture; the code path is the same as for the BASELINE workloads."""
from __future__ import annotations

import os

import numpy as np

from boondock_airband_b200 import abi, synth
from boondock_airband_b200.abi import ChannelCfg, DeviceCfg, EngineCfg

NAMES = ("golden_am_u8", "golden_nfm_s16")
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name: str) -> dict:
    """A fixture's arrays: the outputs in <name>.npz, the input IQ (key "iq") in <name>_iq.npz (two files keep each under 1 MB)."""
    g = dict(np.load(os.path.join(GOLD, name + ".npz")))
    g["iq"] = np.load(os.path.join(GOLD, name + "_iq.npz"))["iq"]
    return g


def build(name: str, with_iq: bool = True):
    if name == "golden_am_u8":
        fs, cf = 256_000, 120_000_000
        ch = [ChannelCfg(freq=cf - 90_000), ChannelCfg(freq=cf - 31_000, bandwidth=5000), ChannelCfg(freq=cf + 27_500, squelch_threshold=-50, ampfactor=1.7),
              ChannelCfg(freq=cf + 77_000, squelch_snr_threshold=6.0, has_iq_outputs=True), ChannelCfg(freq=cf + 110_000, afc=6)]
        dev = DeviceCfg(sample_rate=fs, centerfreq=cf, sample_format="u8", channels=ch)
        cfg = EngineCfg(fft_size=256, wave_rate=8000, devices=[dev], flags=abi.FLAG_TRACE, max_batches_per_step=2)
        iq = synth.synth(dev, 0.66, 101, gate_on=0.22, gate_off=0.09) if with_iq else None
        return cfg, iq
    if name == "golden_nfm_s16":
        fs, cf = 240_000, 162_500_000
        ch = [ChannelCfg(freq=cf - 75_000, modulation="nfm", bandwidth=12_500, ctcss=100.0, notch=100.0),
              ChannelCfg(freq=cf - 25_000, modulation="nfm", bandwidth=12_500, ctcss=100.0, notch=100.0),
              ChannelCfg(freq=cf + 25_000, modulation="nfm", bandwidth=12_500, ctcss=100.0, notch=100.0),
              ChannelCfg(freq=cf + 75_000, modulation="nfm", tau=75, has_iq_outputs=True)]
        dev = DeviceCfg(sample_rate=fs, centerfreq=cf, sample_format="s16", channels=ch)
        cfg = EngineCfg(fft_size=256, wave_rate=16000, devices=[dev], flags=abi.FLAG_TRACE, max_batches_per_step=2)
        iq = synth.synth(dev, 0.78, 102, gate_on=0.62, gate_off=0.1) if with_iq else None
        return cfg, iq
    raise KeyError(name)


# Scenarios on which the restated oracle was compared bit for bit with the reference-built one (oracle/_ref); their outputs
# are recorded as digests in golden/oracle_digests.json (golden/make_oracle_digests.py), so that the comparison keeps
# holding where the reference tree is absent.
def digest_scenarios():
    import scenarios
    return {
        "mixed": lambda: scenarios.mixed_options(0.6),
        "mixed_quadri": lambda: scenarios.mixed_options(0.5, fm_demod=abi.FM_QUADRI_DEMOD),
        "cfg2": lambda: scenarios.cfg2_small(4, 1.0),
        "multi_device": lambda: scenarios.multi_device(0.4),
        "mixed_no_afc": lambda: scenarios.mixed_options(1.2, afc=False),
        "am_stress": lambda: scenarios.am_stress(2.0),
        "afc_walk": lambda: scenarios.afc_walk(1.2),
    }


def oracle_digests(oracle_cls, cfg, streams, ref: bool = False) -> dict:
    """sha256 of everything the oracle hands out per (device, channel): channel constants, audio, decision trace, per-batch
    status, iq_out; and of each device's input bytes."""
    import copy
    import hashlib
    h = lambda b: hashlib.sha256(b).hexdigest()  # noqa: E731
    cfg = copy.copy(cfg)
    cfg.flags |= abi.FLAG_TRACE
    o = oracle_cls(cfg, ref=ref)
    out = {"inputs": [h(np.ascontiguousarray(s).tobytes()) for s in streams], "channels": {}}
    for d, s in enumerate(streams):
        o.feed(d, s)
    for d, dev in enumerate(cfg.devices):
        out["frames_%d" % d] = o.frames(d)
        for c in range(len(dev.channels)):
            rec = {"info": h(bytes(o.channel_info(d, c))), "waveout": h(o.waveout(d, c).tobytes()), "trace": h(o.trace(d, c).tobytes()),
                   "status": h(b"".join(bytes(x) for x in o.status(d, c)))}
            if dev.channels[c].has_iq_outputs:
                rec["iq_out"] = h(o.iq_out(d, c).tobytes())
            out["channels"]["%d/%d" % (d, c)] = rec
    o.close()
    return out
