#!/usr/bin/env python
"""Writes tests/golden/oracle_digests.json: digests of the oracle's outputs on the scenarios of golden_cases.digest_scenarios.
Taken from the reference-built oracle (oracle/_ref) where it exists, else from the restated one, which equals it bit for bit
on these scenarios (tests/test_oracle_pins.py: test_restated_equals_reference_build).

    python tests/golden/make_oracle_digests.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ba_oracle  # noqa: E402
from oracle.ba_oracle import Oracle  # noqa: E402
import golden_cases  # noqa: E402

if __name__ == "__main__":
    ref = ba_oracle.have_ref()
    out = {"source": "oracle/_ref (reference objects)" if ref else "restated oracle"}
    for name, make in golden_cases.digest_scenarios().items():
        cfg, streams = make()
        out[name] = golden_cases.oracle_digests(Oracle, cfg, streams, ref=ref)
        print(name, len(out[name]["channels"]), "channels")
    with open(os.path.join(HERE, "oracle_digests.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
