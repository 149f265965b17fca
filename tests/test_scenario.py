"""Host scenario engine (RINEX-2 reader, orbit/range/iono, code phase, NAV frames, channel
allocation) against the reference's own per-block dumps: every double must be the same bits."""
import os
import subprocess
import sys

import numpy as np
import pytest

import scenario
from scenario import gps

LOC = (35.681298, 139.766247, 10.0)
START = (2024, 1, 7, 2, 0, 0.0)
CASES = {
    "sky12_static_10s_i8": dict(nsat=12, chan=12, secs=10),
    "sky12_static_35s_i8": dict(nsat=12, chan=12, secs=35),
    "sky32_static_10s_i8": dict(nsat=32, chan=32, secs=10),
    "sky12_circle_10s_i16": dict(nsat=12, chan=12, secs=10, motion=True),
    "sky12_rinex3_3s_i8": dict(nsat=12, chan=12, secs=3, v3=True),
    "sky12_pluto_3s_i16": dict(nsat=12, chan=12, secs=3, pluto=True),
    "sky12_target_3s_i8": dict(nsat=12, chan=12, secs=3, target=(1500.5, 33.3, 120.25)),     # -t (gps.c:2348-2357)
}


def make_nav(tmp_path, nsat, v3=False, sets=1):
    nav = tmp_path / ("sky%d.nav" % nsat)
    subprocess.check_call([sys.executable, os.path.join(scenario.ROOT, "oracle", "gen_rinex.py"),
                           "--nsat", str(nsat), "--out", str(nav)] + (["--v3"] if v3 else []) +
                          (["--sets", str(sets)] if sets > 1 else []))
    return str(nav)


# the motion scenarios were dumped with the reference's circle.csv, stored verbatim in tests/golden
CIRCLE = os.path.join(scenario.GOLD, "circle.csv")


@pytest.mark.parametrize("name", list(CASES))
def test_scenario_engine_matches_reference_dump_bit_for_bit(name, tmp_path):
    c = CASES[name]
    g = scenario.load_golden(name)
    want, frames = scenario.golden_chans(g)
    mot = CIRCLE if c.get("motion") else None
    got, nav = gps.scenario(make_nav(tmp_path, c["nsat"], c.get("v3", False)), *LOC, seconds=c["secs"],
                            max_chan=c["chan"], motion_file=mot, start=START, rinex3=c.get("v3", False),
                            pluto_gain=c.get("pluto", False), target=c.get("target"))
    assert got.shape == want.shape
    assert np.array_equal(got["prn"], want["prn"])
    act = want["prn"] > 0
    for f in ("iword", "ibit", "icode"):
        assert np.array_equal(got[f][act], want[f][act]), f
    for f in ("f_carr", "f_code", "code_phase", "gain"):
        a, b = got[f][act].view(np.uint64), want[f][act].view(np.uint64)
        bad = np.nonzero(a != b)[0]
        assert bad.size == 0, (f, bad[:5], got[f][act][bad[:3]], want[f][act][bad[:3]])
    # carrier phase: the engine reports the allocation-time phase (allocateChannel, gps.c:2203-2210)
    assert np.array_equal(got["carr_phase"][0][act[0]], want["carr_phase"][0][act[0]])
    # NAV frames of the active channels
    assert len(nav) == len(frames)
    fidx = g["nav_frame_of_block"]
    assert np.array_equal(got["nav_frame"][:, 0], fidx)
    for b in (0, len(fidx) - 1):
        a = act[b]
        assert np.array_equal(nav[fidx[b]][a], frames[fidx[b]][a])


LOC60 = (60.0, 140.0, 0.0)


def test_reallocation_310s_matches_reference_dump_and_is_thread_invariant(tmp_path, monkeypatch):
    """A satellite rises into a free slot at 240 s, another one sets at 300 s (allocateChannel every 30 s,
    gps.c:2142-2235, 2909): slot occupancy of all 3099 blocks, every parameter around the events and every
    NAV frame against the reference's dump; and the block-parallel builder gives the same bytes for 1 and
    16 threads."""
    g = scenario.load_golden("sky32_lat60_310s_i8")
    nav_file = make_nav(tmp_path, 32)
    runs = []
    for thr in ("1", "16"):
        monkeypatch.setenv("GPSB200_SCENARIO_THREADS", thr)
        runs.append(gps.scenario(nav_file, *LOC60, seconds=310, max_chan=32, start=START))
    (got, nav), (got16, nav16) = runs
    assert got.tobytes() == got16.tobytes() and nav.tobytes() == nav16.tobytes()
    prn = g["prn_of_block"].astype(np.int32)
    assert got.shape == prn.shape and np.array_equal(got["prn"], prn)
    changes = np.nonzero((prn[1:] != prn[:-1]).any(axis=1))[0] + 1
    assert list(changes) == [2400, 3000]                     # the fixture really contains both events
    idx, want = g["chans_idx"], g["chans"]
    for k, b in enumerate(idx):
        act = want["prn"][k] > 0
        for f in ("iword", "ibit", "icode"):
            assert np.array_equal(got[f][b][act], want[f][k][act]), (f, b)
        for f in ("f_carr", "f_code", "code_phase", "gain"):
            assert np.array_equal(got[f][b][act].view(np.uint64), want[f][k][act].view(np.uint64)), (f, b)
    # the slot filled at block 2400 starts from the allocation-time carrier phase (gps.c:2203-2210)
    k = list(idx).index(2400)
    new = (prn[2400] > 0) & (prn[2399] == 0)
    assert new.sum() == 1
    assert np.array_equal(got["carr_phase"][2400][new].view(np.uint64), want["carr_phase"][k][new].view(np.uint64))
    frames, fidx = g["nav_frames"], g["nav_frame_of_block"]
    assert len(nav) == len(frames) and np.array_equal(got["nav_frame"][:, 0], fidx)
    for b in (0, 2399, 2400, 2999, 3000, 3098):
        a = prn[b] > 0
        assert np.array_equal(nav[fidx[b]][a], frames[fidx[b]][a]), b


def test_ephemeris_set_roll_400s_matches_reference_dump(tmp_path):
    """Two ephemeris sets (02:00, 04:00), start 02:55:00: the reference switches to the second set at the
    first 30 s boundary after 03:00:00 (block 3300, gps.c:2890-2905) and rebuilds all subframes. Slot occupancy
    of all 3999 blocks, every parameter around the roll and all 14 NAV frames against the reference's dump."""
    g = scenario.load_golden("sky12_ephroll_400s_i8")
    got, nav = gps.scenario(make_nav(tmp_path, 12, sets=2), *LOC, seconds=400, max_chan=12, start=(2024, 1, 7, 2, 55, 0.0))
    assert np.array_equal(got["prn"], g["prn_of_block"])
    idx, want = g["chans_idx"], g["chans"]
    assert 3300 in idx and 3301 in idx
    for k, b in enumerate(idx):
        act = want["prn"][k] > 0
        for f in ("iword", "ibit", "icode"):
            assert np.array_equal(got[f][b][act], want[f][k][act]), (f, b)
        for f in ("f_carr", "f_code", "code_phase", "gain"):
            assert np.array_equal(got[f][b][act].view(np.uint64), want[f][k][act].view(np.uint64)), (f, b)
    frames, fidx = g["nav_frames"], g["nav_frame_of_block"]
    assert len(nav) == len(frames) == 14 and np.array_equal(got["nav_frame"][:, 0], fidx)
    assert np.array_equal(nav, frames)
    # the frame after the roll really carries new ephemeris words (subframes 1-3), not just a new TOW
    changed = [(frames[i][0] != frames[i - 1][0]).sum() for i in range(1, len(frames))]
    assert max(changed) > 20 and changed.index(max(changed)) + 1 == 12


def test_scenario_errors():
    with pytest.raises(gps.GpsB200Error):
        gps.scenario("/nonexistent.nav", *LOC, seconds=5)


def test_rinex_version_flag_must_match_the_file(tmp_path):
    with pytest.raises(gps.GpsB200Error):
        gps.scenario(make_nav(tmp_path, 12, v3=True), *LOC, seconds=3, start=START)            # v3 file, v2 reader
    with pytest.raises(gps.GpsB200Error):
        gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=3, start=START, rinex3=True)         # v2 file, v3 reader


def test_config3_circle_csv_60s_engine_matches_dump(tmp_path):
    """configs[3] literally: the reference's circle.csv rows (carried in the fixture, re-written with %.17g) for 60 s;
    the first two blocks' parameters are in the fixture, the whole run is compared on the GPU box."""
    g = scenario.load_golden("sky12_circle_60s_i16")
    mot = tmp_path / "circle.csv"
    with open(mot, "w") as f:
        for r in g["motion_rows"]:
            f.write("%.17g,%.17g,%.17g,%.17g\n" % tuple(r))
    got, nav = gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=60, max_chan=12, motion_file=str(mot), start=START)
    assert got.shape == (599, 12)
    for f in ("prn", "iword", "ibit", "icode", "f_carr", "f_code", "code_phase", "gain"):
        assert np.array_equal(got[f][:2], g["chans"][f]), f
    # the re-written rows parse to the same doubles as the original file
    ref, _ = gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=60, max_chan=12, motion_file=CIRCLE, start=START)
    assert got.tobytes() == ref.tobytes()


def test_gzip_compressed_rinex_reads_like_the_plain_file(tmp_path):
    """The reference reads its navigation files through zlib (gzopen/gzgets, gps.c:1147-1157): .gz or plain."""
    import gzip
    import shutil
    for v3 in (False, True):
        nav = make_nav(tmp_path, 12, v3=v3)
        with open(nav, "rb") as fi, gzip.open(nav + ".gz", "wb") as fo:
            shutil.copyfileobj(fi, fo)
        a, na = gps.scenario(nav, *LOC, seconds=2, max_chan=12, start=START, rinex3=v3)
        b, nb = gps.scenario(nav + ".gz", *LOC, seconds=2, max_chan=12, start=START, rinex3=v3)
        assert a.tobytes() == b.tobytes() and na.tobytes() == nb.tobytes()
