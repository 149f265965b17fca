#!/usr/bin/env python3
"""TEST INFRASTRUCTURE: (re)generate tests/golden/*.npz from the reference itself.

Runs only where oracle/Makefile has built the reference binaries (oracle/_ref/ref_*;
that needs the reference sources). For each scenario it runs the UNMODIFIED reference producer
(gps.c, gps_thread_ep) behind the recording FIFO of oracle/ref_harness/ref_dump.c
and stores
  * the per-block channel parameters the sample loop consumed (f_carr, f_code,
    code phase, NAV position, gain, carrier phase at block start, NAV words),
  * CRC-32 digests of every block of the enqueue stream (whole block + 30 parts),
  * a few verbatim blocks,
so that the GPU box (which has no /root/reference) can check the CUDA path and the
C restatement bit for bit against the reference.
Usage: python tests/golden/make_golden.py [names...]
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import refdump  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")
CIRCLE = os.path.join(HERE, "circle.csv")   # the reference's own motion file, stored verbatim
LOC = "35.681298,139.766247,10.0"
START = "2024/01/07,02:00:00"   # = toc of the synthetic ephemerides (avoids date2gps on a zero date)

from motion_track import write_motion  # noqa: E402


SCENARIOS = {
    # name: (nsat, binary, seconds, extra args, keep verbatim blocks)
    "sky12_static_10s_i8": (12, "ref_dump12", 10, [], [0, 98]),
    "sky12_static_35s_i8": (12, "ref_dump12", 35, [], []),
    "sky12_circle_10s_i16": (12, "ref_dump12", 10, ["--iq16", "-m", CIRCLE], [0]),
    "sky32_static_10s_i8": (32, "ref_dump32", 10, [], [0]),
    # BASELINE configs[3]: motion file + --iq16 + 60 s; digests only (parameters come from the scenario engine)
    "sky12_track_60s_i16": (12, "ref_dump12", 60, ["--iq16", "-m", "@MOTION"], []),
    # the same constellation written as RINEX 3 and read by the reference's readRinex3 (-3)
    "sky12_rinex3_3s_i8": (12, "ref_dump12", 3, ["-3"], []),
    # a satellite rises into a free slot at 240 s and another sets at 300 s (allocateChannel, gps.c:2142-2235):
    # 60N 140E, 32 channels, 310 s. Parameters kept only around the events; digests of every block.
    "sky32_lat60_310s_i8": (32, "ref_dump32", 310, [], []),
}
    # two ephemeris sets (02:00 and 04:00), start 02:55:00: the reference rolls to the second set at the first
    # 30 s boundary after 03:00:00 (gps.c:2890-2905) and rebuilds every channel's subframes. 400 s, 12 channels.
SCENARIOS["sky12_ephroll_400s_i8"] = (12, "ref_dump12", 400, [], [])
# BASELINE configs[3] LITERALLY: the reference's own circle.csv, --iq16, 60 s (599 blocks). The motion rows the run
# consumed travel inside the fixture (the GPU box has no /root/reference): tests re-write them with %.17g.
SCENARIOS["sky12_circle_60s_i16"] = (12, "ref_dump12", 60, ["--iq16", "-m", CIRCLE], [])
# ADALM-Pluto flavour of the sample loop: gain x 2 (gps.c:2759-2763), int16 (sdr_pluto.c:107-110)
SCENARIOS["sky12_pluto_3s_i16"] = (12, "ref_dump12", 3, ["--iq16", "--pluto-gain"], [0])
# -t distance,bearing,height: static start point relative to the location (gps.c:2348-2357)
SCENARIOS["sky12_target_3s_i8"] = (12, "ref_dump12", 3, ["-t", "1500.5,33.3,120.25"], [])
LOCS = {"sky32_lat60_310s_i8": "60.0,140.0,0.0"}
STARTS = {"sky12_ephroll_400s_i8": "2024/01/07,02:55:00"}
RINEX_ARGS = {"sky12_ephroll_400s_i8": ["--sets", "2"]}
CHAN_KEEP = {"sky32_lat60_310s_i8": list(range(0, 3)) + list(range(2396, 2405)) + list(range(2996, 3005)) + [3098],
             "sky12_ephroll_400s_i8": list(range(0, 3)) + list(range(3290, 3312)) + [3998]}


def run(name):
    nsat, binary, secs, extra, keep = SCENARIOS[name]
    with tempfile.TemporaryDirectory() as td:
        nav = os.path.join(td, "sky.nav")
        subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "gen_rinex.py"),
                               "--nsat", str(nsat), "--out", nav] + (["--v3"] if "-3" in extra else []) +
                              RINEX_ARGS.get(name, []))
        iq, par = os.path.join(td, "iq.bin"), os.path.join(td, "p.bin")
        if "@MOTION" in extra:
            mot = os.path.join(td, "track.csv")
            write_motion(mot, int(secs * 10))
            extra = [mot if x == "@MOTION" else x for x in extra]
        subprocess.check_call([os.path.join(REF, binary), "-e", nav, "-l", LOCS.get(name, LOC), "-d", str(secs),
                               "-s", STARTS.get(name, START), "--iq", iq, "--params", par] + extra,
                              stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL)
        p = refdump.read_params(par)
        dt = np.int16 if p["sample_size"] == 2 else np.int8
        stream = np.fromfile(iq, dtype=dt)
        ch = p["chans"]
        nblk = ch.shape[0]
        assert stream.size == nblk * 600000, (stream.size, nblk)
        crcs = refdump.block_crcs(stream)
        blocks = stream.reshape(nblk, 600000)
        if name.endswith("60s_i16"):
            ch_keep = ch[:2]            # parameters are recomputed by the scenario engine in the test
            nav_all = refdump.nav_table(p)[:2]
        else:
            ch_keep, nav_all = ch, refdump.nav_table(p)
        extra_out = {}
        if name in CHAN_KEEP:
            idx_keep = np.array(CHAN_KEEP[name], np.int32)
            ch_keep = ch[idx_keep]
            extra_out["chans_idx"] = idx_keep
            extra_out["prn_of_block"] = ch["prn"].astype(np.int8)      # slot occupancy of every block
        out = dict(
            max_chan=np.int32(p["max_chan"]), sample_size=np.int32(p["sample_size"]),
            chans=ch_keep, nav_words=nav_all, crcs=crcs,
            keep_idx=np.array(keep, np.int32),
            keep_blocks=np.stack([blocks[i] for i in keep]) if keep else np.zeros((0, 600000), dt),
            sin512=p["sin512"], cos512=p["cos512"],
            code_prns=np.array(sorted(p["codes"]), np.int32),
            codes=np.stack([p["codes"][k] for k in sorted(p["codes"])]),
        )
        # NAV words change every 300 blocks: store one copy per distinct frame.
        nw = out.pop("nav_words")
        frames, idx = [], np.zeros(nblk, np.int32)
        for b in range(nw.shape[0]):
            if not frames or not np.array_equal(frames[-1], nw[b]):
                frames.append(nw[b])
            idx[b] = len(frames) - 1
        out["nav_frames"] = np.stack(frames)
        out["nav_frame_of_block"] = idx
        out.update(extra_out)
        if CIRCLE in extra:
            rows = np.loadtxt(CIRCLE, delimiter=",")
            out["motion_rows"] = rows[:int(secs * 10)]
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        print(name, "blocks", nblk, "chan", p["max_chan"], "frames", len(frames),
              "active", int((ch["prn"][0] > 0).sum()))


def run_crc_only(name, nsat, binary, secs, crc_file=None):
    """Long runs: only the CRC-32 of every enqueued block is kept (ref_dump --crc); parameters come from
    the scenario engine in the test. crc_file: reuse the output of an earlier (background) run of exactly
    this command line."""
    with tempfile.TemporaryDirectory() as td:
        if crc_file is None:
            nav = os.path.join(td, "sky.nav")
            subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "gen_rinex.py"),
                                   "--nsat", str(nsat), "--out", nav])
            crc_file = os.path.join(td, "crc.bin")
            subprocess.check_call([os.path.join(REF, binary), "-e", nav, "-l", LOC, "-d", str(secs), "-s", START,
                                   "--crc", crc_file], stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL)
        crcs = np.fromfile(crc_file, dtype="<u4")
    assert crcs.size == int(secs * 10 + 0.5) - 1, crcs.size
    np.savez_compressed(os.path.join(HERE, name + ".npz"), crcs=crcs, max_chan=np.int32(nsat), sample_size=np.int32(1),
                        seconds=np.int32(secs))
    print(name, "blocks", crcs.size)


# BASELINE configs[4]: 32 channels, int8, 3600 s (35 999 blocks). The -O2 build of the unmodified reference
# (byte-identical output, see oracle/Makefile) needs ~25 min of one CPU for it.
CRC_ONLY = {"sky32_static_3600s_i8": (32, "ref_run32_fast", 3600)}


def run_stock(name, nsat, binary, secs):
    """The reference program exactly as shipped (own fifo.c / sdr_iqfile.c): CRC-32 of every block of the
    iqdata.bin it writes."""
    with tempfile.TemporaryDirectory() as td:
        nav = os.path.join(td, "sky.nav")
        subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "gen_rinex.py"),
                               "--nsat", str(nsat), "--out", nav])
        subprocess.check_call([os.path.join(REF, binary), "-e", nav, "-l", LOC, "-d", str(secs)], cwd=td,
                              stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL)
        crcs = refdump.block_crcs(np.fromfile(os.path.join(td, "iqdata.bin"), dtype=np.int8))[:, 0]
    np.savez_compressed(os.path.join(HERE, name + ".npz"), crcs=crcs, max_chan=np.int32(nsat), sample_size=np.int32(1),
                        seconds=np.int32(secs))
    print(name, "blocks", crcs.size)


# configs[1] through the stock program: its FIFO loses buffers 1..6 (fifo.c:163-168)
STOCK = {"sky12_static_10s_stock_iqfile": (12, "ref_stock12", 10)}


if __name__ == "__main__":
    args = sys.argv[1:]
    crc_file = None
    if "--crc-file" in args:
        i = args.index("--crc-file")
        crc_file = args[i + 1]
        del args[i:i + 2]
    for n in (args or list(SCENARIOS) + list(CRC_ONLY) + list(STOCK)):
        if n in CRC_ONLY:
            run_crc_only(n, *CRC_ONLY[n], crc_file=crc_file)
        elif n in STOCK:
            run_stock(n, *STOCK[n])
        else:
            run(n)
