#!/usr/bin/env python3
"""TEST INFRASTRUCTURE: (re)generate the fixtures of the reference's INTEGER carrier build (gps.h:17 without
`#define FLOAT_CARR_PHASE`), tests/golden/*_u32.npz, with the same recorder and record layout as make_golden.py.

The reference binaries come from oracle/u32.mk (oracle/_ref/ref_*_u32; that needs the reference sources). The dumped
carr_phase of these fixtures is the reference's unsigned 32-bit accumulator (an integer-valued double).
Usage: python tests/golden/make_golden_u32.py [names...]
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402

SCENARIOS = {
    # BASELINE configs[1] on the integer build: block 0 verbatim (the other blocks, 98 included, by their whole-block
    # and 30 part CRCs: a second verbatim block would take the fixture past 1 MB)
    "sky12_static_10s_i8_u32": (12, "ref_dump12_u32", 10, [], [0]),
    "sky32_static_10s_i8_u32": (32, "ref_dump32_u32", 10, [], [0]),
    # configs[3] on the integer build: the reference's circle.csv, --iq16, 60 s
    "sky12_circle_60s_i16_u32": (12, "ref_dump12_u32", 60, ["--iq16", "-m", mg.CIRCLE], []),
    # 60N 140E, 32 channels, 310 s: a satellite rises into a free slot at 240 s and another sets at 300 s
    "sky32_lat60_310s_i8_u32": (32, "ref_dump32_u32", 310, [], []),
}
CRC_ONLY = {"sky32_static_600s_i8_u32": (32, "ref_run32_u32_fast", 600)}

mg.SCENARIOS.update(SCENARIOS)
mg.LOCS["sky32_lat60_310s_i8_u32"] = mg.LOCS["sky32_lat60_310s_i8"]
mg.CHAN_KEEP["sky32_lat60_310s_i8_u32"] = mg.CHAN_KEEP["sky32_lat60_310s_i8"]

if __name__ == "__main__":
    for n in sys.argv[1:] or list(SCENARIOS) + list(CRC_ONLY):
        if n in CRC_ONLY:
            mg.run_crc_only(n, *CRC_ONLY[n])
        else:
            mg.run(n)
