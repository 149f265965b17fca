"""Almanac pages from a SEM almanac file (scenario config `almanac_file`, Python `scenario(..., almanac=)`, CLI
`--almanac`): the reference fills subframe 4 pages 2-5 / 7-10 (PRN 25-32), subframe 5 pages 1-24 (PRN 1-24) and the
toa/WNa of subframe 5 page 25 from its almanac.sem (almanac.c:73-184, gps.c:772-884, 2614-2651).

Fixtures (tests/golden/*_alm*.npz, make_golden_alm.py): the reference run with its almanac enabled; each stores the
SEM text it read, the NAV frames, the PRN of every slot and block, and the CRC-32 of every block.
CPU: the engine's NAV frames against the reference's for every fixture and every edge-case file of the SEM reader,
channel records untouched by the almanac, the start-time check, and the oracle on blocks that carry almanac pages.
GPU: whole streams with almanac pages through the library (both carrier NCOs) and the CLI on 1 and 2 GPUs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import scenario
from scenario import gps

LOC = (35.681298, 139.766247, 10.0)
LOC60 = (60.0, 140.0, 0.0)
START = (2024, 1, 7, 2, 0, 0.0)
START_ROLL = (2024, 1, 7, 2, 55, 0.0)
EDGES = "sky12_static_35s_alm_edges"
sys.path.insert(0, os.path.join(scenario.ROOT, "oracle"))
import gen_almanac  # noqa: E402

# fixture: (channels, seconds, location, start, ephemeris sets, carrier)
RUNS = {
    "sky12_ephroll_760s_i8_alm": (12, 760, LOC, START_ROLL, 2, "fp64"),
    "sky32_lat60_310s_i8_alm": (32, 310, LOC60, START, 1, "fp64"),
    "sky12_static_65s_i8_u32_alm": (12, 65, LOC, START, 1, "u32"),
}


def make_nav(tmp_path, nsat, sets=1):
    nav = tmp_path / ("sky%d_%d.nav" % (nsat, sets))
    if not nav.exists():
        subprocess.check_call([sys.executable, os.path.join(scenario.ROOT, "oracle", "gen_rinex.py"),
                               "--nsat", str(nsat), "--out", str(nav), "--sets", str(sets)])
    return str(nav)


def write_sem(tmp_path, data, name="almanac.sem"):
    """The SEM text stored in a fixture (uint8), or a str, written byte for byte."""
    p = tmp_path / name
    p.write_bytes(data.tobytes() if isinstance(data, np.ndarray) else data.encode())
    return str(p)


def run_engine(name, tmp_path, almanac=True, carrier=None):
    g = scenario.load_golden(name)
    nsat, secs, loc, start, sets, carr = RUNS[name]
    sem = write_sem(tmp_path, g["sem"]) if almanac else None
    ch, nav = gps.scenario(make_nav(tmp_path, nsat, sets), *loc, seconds=secs, max_chan=nsat, start=start,
                           carrier=carrier or carr, almanac=sem)
    return g, ch, nav


def assert_nav_equal(ch, nav, prn_of_block, want_frames, want_idx, what):
    """Every active slot of every block carries the reference's words."""
    assert np.array_equal(ch["prn"], prn_of_block), what
    pairs = np.unique(np.stack([ch["nav_frame"][:, 0], want_idx], 1), axis=0)
    for fe, fr in pairs:
        blocks = np.nonzero((ch["nav_frame"][:, 0] == fe) & (want_idx == fr))[0]
        active = np.nonzero(prn_of_block[blocks[0]] > 0)[0]
        assert np.array_equal(nav[fe][active], want_frames[fr][active]), (what, int(blocks[0]), int(fe), int(fr))


# ---- CPU ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(RUNS))
def test_engine_nav_frames_equal_the_reference(name, tmp_path):
    g, ch, nav = run_engine(name, tmp_path)
    assert ch.shape[0] == g["crcs"].size
    assert_nav_equal(ch, nav, g["prn_of_block"], g["nav_frames"], g["nav_frame_of_block"], name)
    if name.startswith("sky12_ephroll"):        # all 25 pages of subframes 4 and 5 in every slot
        assert len(nav) == 26


@pytest.mark.parametrize("case", gen_almanac.CASES)
def test_engine_reads_edge_case_files_like_the_reference(case, tmp_path):
    g = scenario.load_golden(EDGES)
    ch, nav = gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=35, start=START,
                           almanac=write_sem(tmp_path, g[case + "/sem"]))
    assert_nav_equal(ch, nav, g[case + "/prn_of_block"], g[case + "/nav_frames"], g[case + "/nav_frame_of_block"], case)


def test_fixture_sem_texts_are_the_generators():
    """The stored SEM texts are what oracle/gen_almanac.py writes (the fixtures and the generator agree)."""
    assert scenario.load_golden("sky12_ephroll_760s_i8_alm")["sem"].tobytes() == gen_almanac.text().encode()
    g = scenario.load_golden(EDGES)
    for case in gen_almanac.CASES:
        assert g[case + "/sem"].tobytes() == gen_almanac.text(case).encode(), case


def test_fixture_values_separate_the_literal_scales_from_true_powers_of_two():
    """PRN 1's fields sit a few ulps below multiples of their scales, so that dividing by gps.h's POW2_M38 / POW2_M23
    literals and by the true powers of two truncate to different integers (the fixtures pin the literals)."""
    r = gen_almanac.records()[1]
    for f, lit in (("omegadot", 3.63797880709171e-012), ("af1", 3.63797880709171e-012), ("omega0", 1.19209289550781e-007),
                   ("aop", 1.19209289550781e-007), ("m0", 1.19209289550781e-007)):
        assert int(r[f] / lit) != int(r[f] / gen_almanac.SCALE[f]), f
    signed = ("delta_i", "omegadot", "omega0", "aop", "m0", "af0", "af1")
    recs = gen_almanac.records().values()
    assert all(any(rec[f] < 0 for rec in recs) for f in signed)


def test_almanac_changes_only_nav_words(tmp_path):
    _, ch_a, nav_a = run_engine("sky12_ephroll_760s_i8_alm", tmp_path)
    _, ch_n, nav_n = run_engine("sky12_ephroll_760s_i8_alm", tmp_path, almanac=False)
    assert ch_a.tobytes() == ch_n.tobytes()
    assert nav_a.shape == nav_n.shape and not np.array_equal(nav_a, nav_n)
    # subframes 1-3 (words 10..39 of a frame) are the same; only the words of subframes 4 and 5 differ
    assert np.array_equal(nav_a[:, :, 10:40], nav_n[:, :, 10:40])


def test_dropped_almanac_equals_no_almanac(tmp_path):
    """A parse error before the end of the file drops the whole almanac: every page is a dummy page."""
    g = scenario.load_golden(EDGES)
    nav_file = make_nav(tmp_path, 12)
    ch_d, nav_d = gps.scenario(nav_file, *LOC, seconds=35, start=START, almanac=write_sem(tmp_path, g["badline/sem"]))
    ch_n, nav_n = gps.scenario(nav_file, *LOC, seconds=35, start=START)
    assert ch_d.tobytes() == ch_n.tobytes() and nav_d.tobytes() == nav_n.tobytes()


def old_sem():
    return gen_almanac.text(week=gen_almanac.WEEK - 5)        # toa 5 weeks before the start (minus 15 h)


def test_almanac_toa_more_than_4_weeks_from_the_start_is_an_error(tmp_path):
    with pytest.raises(gps.GpsB200Error, match="almanac"):
        gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=3, start=START, almanac=write_sem(tmp_path, old_sem()))
    # 4 weeks minus 15 h earlier is still accepted
    gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=3, start=START,
                 almanac=write_sem(tmp_path, gen_almanac.text(week=gen_almanac.WEEK - 4), "a4.sem"))


@pytest.mark.ref
def test_reference_writes_no_block_for_that_almanac(tmp_path):
    exe = os.path.join(scenario.ROOT, "oracle", "_ref", "ref_dump12_alm")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_dump12_alm not built (needs the reference sources)")
    write_sem(tmp_path, old_sem())
    r = subprocess.run([exe, "--almanac", "-e", make_nav(tmp_path, 12), "-l", "%r,%r,%r" % LOC, "-d", "3",
                        "-s", "2024/01/07,02:00:00"], cwd=tmp_path, capture_output=True, text=True)
    assert json.loads(r.stdout.strip().splitlines()[-1])["blocks"] == 0


def test_missing_almanac_file_is_an_error(tmp_path):
    with pytest.raises(gps.GpsB200Error, match="almanac"):
        gps.scenario(make_nav(tmp_path, 12), *LOC, seconds=3, start=START, almanac=str(tmp_path / "none.sem"))


def test_oracle_reproduces_blocks_with_almanac_pages(tmp_path):
    """The C oracle on the engine's records and NAV frames, at blocks that transmit almanac words in every slot: frame 1
    (subframe 4 page 2 = PRN 25, subframe 5 page 2 = PRN 2), frame 11 after the ephemeris roll at block 3300 (subframe 5
    page 12) and frame 24 (subframe 5 page 25, the almanac's toa/WNa). Each block starts from the exactly chained
    carrier phase."""
    g, ch, nav = run_engine("sky12_ephroll_760s_i8_alm", tmp_path)
    _, _, nav_none = run_engine("sky12_ephroll_760s_i8_alm", tmp_path, almanac=False)
    assert (ch["prn"] == ch["prn"][0]).all()            # static sky: the same 12 satellites throughout
    phase, b0 = None, 0
    for b in (500, 560, 3560, 7460):
        f, slots = ch["nav_frame"][b, 0], np.arange(ch.shape[1])
        iw = ch["iword"][b]
        assert (nav[f, slots, iw] != nav_none[f, slots, iw]).all(), b      # the word in transit is an almanac word
        phase = gps.carrier_chain(ch[b0:b], phase_in=phase)
        row = ch[b:b + 1].copy()
        row["carr_phase"][0] = phase
        out, _ = scenario.oracle_run(row, nav, 1)
        assert scenario.crc_blocks(out)[0] == g["crcs"][b], b
        b0 = b


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def synth_crcs(ch, nav, carrier="fp64", per_call=3000):
    """CRC-32 of every block, consecutive calls chained by their outgoing carrier phases."""
    nblk, nchan = ch.shape
    crcs, cp = [], None
    with gps.Context(nchan, min(per_call, nblk), max_nav_frames=len(nav), carrier=carrier) as ctx:
        ctx.set_nav_frames(nav)
        for b0 in range(0, nblk, per_call):
            part = ch[b0:b0 + per_call].copy()
            if cp is not None:
                cont = (part["prn"][0] > 0) & (part["prn"][0] == ch["prn"][b0 - 1])
                part["carr_phase"][0][cont] = cp[cont]
            out, cp = ctx.synth_blocks(part, 1)
            crcs.append(scenario.crc_blocks(out))
    return np.concatenate(crcs)


def assert_crcs(crc, want, what):
    assert crc.size == want.size, (what, crc.size, want.size)
    bad = np.nonzero(crc != want)[0]
    assert bad.size == 0, "%s: %d/%d blocks differ, first %s" % (what, bad.size, crc.size, bad[:5])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RUNS))
def test_streams_with_almanac_pages_equal_the_reference(name, tmp_path):
    g, ch, nav = run_engine(name, tmp_path)
    assert_crcs(synth_crcs(ch, nav, RUNS[name][5]), g["crcs"], name)


@pytest.mark.gpu
def test_cli_almanac_writes_the_reference_stream(tmp_path):
    """gpsb200-sim --almanac, 65 s from the inputs of the 760 s fixture: its first 649 blocks; --gpus 2 where two
    devices are visible."""
    import torch
    exe = os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "gpsb200-sim")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "csrc")])
    g = scenario.load_golden("sky12_ephroll_760s_i8_alm")
    sem = write_sem(tmp_path, g["sem"])
    cmd = [exe, "-e", make_nav(tmp_path, 12, 2), "-l", "%r,%r,%r" % LOC, "-s", "2024/01/07,02:55:00", "-d", "65",
           "--almanac", sem]
    for n in [1] + ([2] if torch.cuda.device_count() >= 2 else []):
        out = tmp_path / ("iq_%d.bin" % n)
        r = subprocess.run(cmd + ["--gpus", str(n), "-o", str(out)], capture_output=True, text=True, check=True)
        assert "no almanac pages" not in r.stderr
        s = np.fromfile(out, dtype=np.int8)
        assert s.size == 649 * gps.BLOCK_ELEMS
        assert_crcs(scenario.crc_blocks(s), g["crcs"][:649], "cli --gpus %d" % n)
