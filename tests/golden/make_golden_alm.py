#!/usr/bin/env python3
"""TEST INFRASTRUCTURE: (re)generate the almanac fixtures, tests/golden/*_alm*.npz, from the reference itself.

The reference producer runs behind the recorder of make_golden.py with its almanac enabled (oracle/alm.mk builds
oracle/_ref/ref_dump*_alm, switch --almanac; that needs the reference sources). It reads almanac.sem from its working
directory, so every run happens in a temporary directory holding the SEM file of oracle/gen_almanac.py. Each fixture
stores that SEM text verbatim (`sem`, uint8), so the tests rebuild the exact input without running the generator,
plus the NAV frames, the frame of every block, the PRN of every slot and block and the CRC-32 of every whole block.
Per-block channel parameters are left out: they do not depend on the almanac, and the tests compare the engine's
records with and without it.
Usage: python tests/golden/make_golden_alm.py [names...]
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402

ROOT = mg.ROOT
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import gen_almanac  # noqa: E402
import refdump  # noqa: E402

# name: (nsat, binary, seconds, location, start, ephemeris sets, almanac case)
SCENARIOS = {
    # two ephemeris sets, start 02:55:00, 760 s: 26 NAV frames, so all 25 pages of subframes 4 and 5 pass through every
    # slot, and the ephemeris roll at block 3300 rebuilds the subframes with the almanac
    "sky12_ephroll_760s_i8_alm": (12, "ref_dump12_alm", 760, mg.LOC, "2024/01/07,02:55:00", 2, None),
    # 60N 140E, 32 channels: a satellite rises into a free slot at 240 s (starting at page 0 while the other slots are
    # at pages 8-9) and another sets at 300 s
    "sky32_lat60_310s_i8_alm": (32, "ref_dump32_alm", 310, "60.0,140.0,0.0", mg.START, 1, None),
    # the integer carrier build (gps.h:17 without FLOAT_CARR_PHASE)
    "sky12_static_65s_i8_u32_alm": (12, "ref_dump12_u32_alm", 65, mg.LOC, mg.START, 1, None),
}
# one 35 s run per edge-case SEM file, all in one fixture (keys prefixed with the case name)
EDGES = "sky12_static_35s_alm_edges"


def run_one(nsat, binary, secs, loc, start, sets, case):
    """-> dict(sem, crcs, nav_frames, nav_frame_of_block, prn_of_block, max_chan, sample_size)"""
    sem = gen_almanac.text(case)
    with tempfile.TemporaryDirectory() as td:
        nav = os.path.join(td, "sky.nav")
        subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "gen_rinex.py"), "--nsat", str(nsat),
                               "--out", nav, "--sets", str(sets)])
        with open(os.path.join(td, "almanac.sem"), "w", newline="") as f:
            f.write(sem)
        crc, par = os.path.join(td, "crc.bin"), os.path.join(td, "p.bin")
        subprocess.check_call([os.path.join(mg.REF, binary), "--almanac", "-e", nav, "-l", loc, "-d", str(secs),
                               "-s", start, "--crc", crc, "--params", par], cwd=td,
                              stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL)
        p = refdump.read_params(par)
        crcs = np.fromfile(crc, dtype="<u4")
    ch = p["chans"]
    assert crcs.size == ch.shape[0] == int(secs * 10 + 0.5) - 1, (crcs.size, ch.shape)
    nw = refdump.nav_table(p)
    frames, idx = [], np.zeros(nw.shape[0], np.int32)
    for b in range(nw.shape[0]):
        if not frames or not np.array_equal(frames[-1], nw[b]):
            frames.append(nw[b])
        idx[b] = len(frames) - 1
    return dict(sem=np.frombuffer(sem.encode(), np.uint8), crcs=crcs, nav_frames=np.stack(frames),
                nav_frame_of_block=idx, prn_of_block=ch["prn"].astype(np.int8),
                max_chan=np.int32(p["max_chan"]), sample_size=np.int32(p["sample_size"]))


def run(name):
    nsat, binary, secs, loc, start, sets, case = SCENARIOS[name]
    out = run_one(nsat, binary, secs, loc, start, sets, case)
    out.update(seconds=np.int32(secs), loc=np.array([float(v) for v in loc.split(",")]), start=np.array(start),
               sets=np.int32(sets))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "blocks", out["crcs"].size, "frames", out["nav_frames"].shape[0])


def run_edges():
    out = dict(cases=np.array(gen_almanac.CASES), seconds=np.int32(35))
    for case in gen_almanac.CASES:
        for k, v in run_one(12, "ref_dump12_alm", 35, mg.LOC, mg.START, 1, case).items():
            out[case + "/" + k] = v
        print(EDGES, case, "frames", out[case + "/nav_frames"].shape[0])
    np.savez_compressed(os.path.join(HERE, EDGES + ".npz"), **out)


if __name__ == "__main__":
    for n in sys.argv[1:] or list(SCENARIOS) + [EDGES]:
        if n == EDGES:
            run_edges()
        else:
            run(n)
