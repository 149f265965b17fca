"""GPU parity tests: the CUDA path, called through the C ABI of libgpsb200.so,
against (a) digests of the reference's own output (tests/golden, produced by the
unmodified reference) and (b) the CPU oracle on seeded synthetic parameters.
Bit-exact everywhere: the path is integer output from exactly reproduced FP64 NCOs."""
import numpy as np
import pytest

import scenario
from scenario import gps

pytestmark = pytest.mark.gpu


def run_golden(name, nblocks=None, run_samples=0):
    g = scenario.load_golden(name)
    ch, frames = scenario.golden_chans(g, nblocks)
    nblk, nchan = ch.shape
    ss = int(g["sample_size"])
    with gps.Context(nchan, nblk, max_nav_frames=len(frames), run_samples=run_samples) as ctx:
        ctx.set_nav_frames(frames)
        out, cp = ctx.synth_blocks(ch, ss)
    crc = scenario.crc_blocks(out)
    want = g["crcs"][:nblk, 0]
    bad = np.nonzero(crc != want)[0]
    assert bad.size == 0, "%s: %d/%d blocks differ from the reference, first %s" % (name, bad.size, nblk, bad[:5])
    for i, blk in zip(g["keep_idx"], g["keep_blocks"]):
        if i < nblk:
            assert np.array_equal(out[i * gps.BLOCK_ELEMS:(i + 1) * gps.BLOCK_ELEMS], blk)
    return g, out


def test_config1_sky12_static_10s_int8_matches_reference_stream():
    g, out = run_golden("sky12_static_10s_i8")
    # the stock program's iqdata.bin is this stream without blocks 1..6 (fifo.c:163-168)
    assert out.size == 99 * gps.BLOCK_ELEMS


def test_sky32_static_10s_int8_matches_reference_stream():
    run_golden("sky32_static_10s_i8")


def test_config3_motion_int16_matches_reference_stream():
    run_golden("sky12_circle_10s_i16")


def test_nav_frame_roll_and_35s_chain_matches_reference_stream():
    run_golden("sky12_static_35s_i8")


@pytest.mark.parametrize("run_samples", [800, 4000, 12000])
def test_other_run_lengths_give_identical_output(run_samples):
    run_golden("sky12_static_10s_i8", nblocks=12, run_samples=run_samples)


@pytest.mark.parametrize("nchan,ss", [(1, 1), (5, 2), (8, 1), (9, 1), (16, 2), (17, 1), (32, 1), (32, 2)])
def test_synthetic_vs_oracle(nchan, ss):
    ch, nav = scenario.synthetic_chans(3, nchan, seed=100 + nchan)
    want, carr = scenario.oracle_run(ch, nav, ss)
    with gps.Context(nchan, 3) as ctx:
        ctx.set_nav_frames(nav)
        out, cp = ctx.synth_blocks(ch, ss)
    assert np.array_equal(out, want)
    assert np.array_equal(cp, carr)


def test_edge_cases_vs_oracle():
    # unused slots, tiny and zero Doppler, negative Doppler, gains below 0.5 (table entries truncate to 0),
    # carrier phase close to the wrap, code phase close to 1023
    ch, nav = scenario.synthetic_chans(2, 12, seed=7, active=[1, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1, 0])
    ch["f_carr"][:, 0] = 0.0
    ch["f_carr"][:, 1] = 1e-3
    ch["f_carr"][:, 3] = -4999.5
    ch["f_carr"][:, 4] = 0.37
    ch["f_carr"][:, 5] = -0.002
    ch["f_code"] = 1.023e6 + ch["f_carr"] / 1540.0
    ch["gain"][:, 7] = 0.004
    ch["gain"][:, 8] = 0.3
    ch["carr_phase"][0, 9] = 1.0 - 2.0 ** -53
    ch["carr_phase"][0, 3] = 2.0 ** -60
    ch["code_phase"][:, 10] = np.nextafter(1023.0, 0.0)
    for ss in (1, 2):
        want, carr = scenario.oracle_run(ch, nav, ss)
        with gps.Context(12, 2) as ctx:
            ctx.set_nav_frames(nav)
            out, cp = ctx.synth_blocks(ch, ss)
        assert np.array_equal(out, want)
        assert np.array_equal(cp, carr)


def test_split_calls_equal_one_call_and_device_path_equals_host_path():
    import torch
    ch, nav = scenario.synthetic_chans(6, 32, seed=3)
    with gps.Context(32, 6) as ctx:
        ctx.set_nav_frames(nav)
        whole, cp = ctx.synth_blocks(ch, 1)
        a, cpa = ctx.synth_blocks(ch[:2], 1)
        rest = ch[2:].copy()
        rest["carr_phase"][0] = cpa
        b, cpb = ctx.synth_blocks(rest, 1)
        assert np.array_equal(np.concatenate([a, b]), whole)
        assert np.array_equal(cpb, cp)
        dev = torch.empty(6 * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
        cpd = ctx.synth_blocks_device(ch, 1, dev.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(dev.cpu().numpy(), whole)
        assert np.array_equal(cpd, cp)
        dev.zero_()
        ctx.replay_device(dev.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(dev.cpu().numpy(), whole)


def test_int16_linearity_over_channels_full_block():
    # size-independent property: before quantisation the stream is a sum over channels
    ch, nav = scenario.synthetic_chans(2, 32, seed=11)
    with gps.Context(32, 2) as ctx:
        ctx.set_nav_frames(nav)
        full, _ = ctx.synth_blocks(ch, 2)
        lo, hi = ch.copy(), ch.copy()
        lo["prn"][:, 16:] = 0
        hi["prn"][:, :16] = 0
        a, _ = ctx.synth_blocks(lo, 2)
        b, _ = ctx.synth_blocks(hi, 2)
    assert np.array_equal(a.astype(np.int32) + b.astype(np.int32), full.astype(np.int32))
    q = ((full.astype(np.int32) >> 4) & 0xFF).astype(np.uint8).view(np.int8)
    with gps.Context(32, 2) as ctx:
        ctx.set_nav_frames(nav)
        i8, _ = ctx.synth_blocks(ch, 1)
    assert np.array_equal(i8, q)


def test_errors_are_loud():
    ch, nav = scenario.synthetic_chans(1, 4, seed=5)
    with gps.Context(4, 1) as ctx:
        ctx.set_nav_frames(nav)
        bad = ch.copy()
        bad["gain"] = 40.0
        with pytest.raises(gps.GpsB200Error) as e:
            ctx.synth_blocks(bad, 1)
        assert e.value.code == -3
        bad = ch.copy()
        bad["code_phase"][0, 0] = 1023.0
        with pytest.raises(gps.GpsB200Error) as e:
            ctx.synth_blocks(bad, 1)
        assert e.value.code == -1
        with pytest.raises(gps.GpsB200Error):
            ctx.synth_blocks(np.concatenate([ch, ch]), 1)      # nblk > max_blocks
        for field, val in (("f_code", 2.0e6), ("f_carr", 3.1e6), ("f_carr", float("nan"))):
            bad = ch.copy()
            bad[field][0, 1] = val
            with pytest.raises(gps.GpsB200Error) as e:
                ctx.synth_blocks(bad, 1)
            assert e.value.code == -1


def test_full_size_300s_32ch_int8_properties():
    """BASELINE configs[2] at full size (2999 blocks x 32 channels = 899.7 Msamples, 1.8 GB):
    the segmented host-destination path equals the single-segment device path byte for byte,
    and sampled blocks equal the CPU oracle started from carrier phases obtained by the
    SEQUENTIAL exact chain (gpsb200_carrier_chain) -- i.e. independently of the speculative
    parallel-in-time chain the pipeline uses."""
    import torch
    import zlib
    nblk, nchan = 2999, 32
    ch, nav = gps.synthetic_chans(nblk, nchan, seed=2024)
    with gps.Context(nchan, nblk) as ctx:
        ctx.set_nav_frames(nav)
        host = torch.empty(nblk * gps.BLOCK_ELEMS, dtype=torch.int8, pin_memory=True)
        out, cp, st = ctx.synth_blocks(ch, 1, out=host.numpy(), want_stats=True)
        dev = torch.empty(nblk * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
        cpd = ctx.synth_blocks_device(ch, 1, dev.data_ptr())
        torch.cuda.synchronize()
        assert torch.equal(host.cuda(), dev)
        assert np.array_equal(cp, cpd)
    assert st.chain_fallbacks < 0.01 * nblk * nchan
    assert np.array_equal(cp, gps.carrier_chain(ch, threads=8))          # speculative == sequential chain
    for b in (1, 1234, 2998):
        start = gps.carrier_chain(ch[:b], threads=8)
        one = ch[b:b + 1].copy()
        one["carr_phase"][0] = start
        want, _ = scenario.oracle_run(one, nav, 1)
        got = out[b * gps.BLOCK_ELEMS:(b + 1) * gps.BLOCK_ELEMS]
        assert zlib.crc32(got.tobytes()) == zlib.crc32(want.tobytes()), b


def _nav_file(tmp_path, nsat):
    import subprocess
    import sys
    import os
    nav = tmp_path / ("sky%d.nav" % nsat)
    subprocess.check_call([sys.executable, os.path.join(scenario.ROOT, "oracle", "gen_rinex.py"),
                           "--nsat", str(nsat), "--out", str(nav)])
    return str(nav)


@pytest.mark.parametrize("name,nsat,chan,secs", [("sky12_static_10s_i8", 12, 12, 10), ("sky32_static_10s_i8", 32, 32, 10),
                                                 ("sky12_static_35s_i8", 12, 12, 35)])
def test_config1_from_rinex_file_to_reference_stream(name, nsat, chan, secs, tmp_path):
    """BASELINE configs[1] literally: RINEX + location + start time in, IQ stream out, no
    reference-produced parameter anywhere -- compared with the reference's stream."""
    g = scenario.load_golden(name)
    ch, nav = gps.scenario(_nav_file(tmp_path, nsat), 35.681298, 139.766247, 10.0, seconds=secs, max_chan=chan,
                           start=(2024, 1, 7, 2, 0, 0.0))
    with gps.Context(chan, ch.shape[0], max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 1)
    assert np.array_equal(scenario.crc_blocks(out), g["crcs"][:, 0])


def test_reallocation_310s_from_rinex_file_to_reference_stream(tmp_path):
    """60N 140E, 32 channels, 310 s: a satellite rises into a free slot at 240 s (fresh carrier phase, NAV frame
    built for the new slot) and another sets at 300 s. RINEX in, all 3099 blocks equal to the reference's stream."""
    g = scenario.load_golden("sky32_lat60_310s_i8")
    ch, nav = gps.scenario(_nav_file(tmp_path, 32), 60.0, 140.0, 0.0, seconds=310, max_chan=32, start=(2024, 1, 7, 2, 0, 0.0))
    assert ch.shape[0] == 3099
    with gps.Context(32, ch.shape[0], max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 1)
    bad = np.nonzero(scenario.crc_blocks(out) != g["crcs"][:, 0])[0]
    assert bad.size == 0, bad[:10]


def test_ephemeris_roll_400s_from_rinex_file_to_reference_stream(tmp_path):
    """Two ephemeris sets in the RINEX file, start 02:55:00, 400 s: the set roll at block 3300 (new subframes, a range
    step between the sets). RINEX in, all 3999 blocks equal to the reference's stream."""
    import os
    import subprocess
    import sys
    g = scenario.load_golden("sky12_ephroll_400s_i8")
    nav_file = tmp_path / "sky12x2.nav"
    subprocess.check_call([sys.executable, os.path.join(scenario.ROOT, "oracle", "gen_rinex.py"), "--nsat", "12", "--sets", "2",
                           "--out", str(nav_file)])
    ch, nav = gps.scenario(str(nav_file), 35.681298, 139.766247, 10.0, seconds=400, max_chan=12, start=(2024, 1, 7, 2, 55, 0.0))
    assert ch.shape[0] == 3999
    with gps.Context(12, ch.shape[0], max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 1)
    bad = np.nonzero(scenario.crc_blocks(out) != g["crcs"][:, 0])[0]
    assert bad.size == 0, bad[:10]


def test_cli_writes_reference_iqfile_and_stock_compat_file(tmp_path):
    import os
    import subprocess
    import zlib
    exe = os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "gpsb200-sim")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "csrc")])
    nav = _nav_file(tmp_path, 12)
    g = scenario.load_golden("sky12_static_10s_i8")
    for extra, keep in (([], list(range(99))), (["--compat-drop"], [0] + list(range(7, 99)))):
        out = tmp_path / ("iq%d.bin" % len(extra))
        subprocess.check_call([exe, "-e", nav, "-l", "35.681298,139.766247,10.0", "-d", "10",
                               "-s", "2024/01/07,02:00:00", "-o", str(out)] + extra)
        s = np.fromfile(out, dtype=np.int8)
        assert s.size == len(keep) * gps.BLOCK_ELEMS, (extra, s.size)
        for row, b in zip(s.reshape(len(keep), gps.BLOCK_ELEMS), keep):
            assert zlib.crc32(row.tobytes()) == g["crcs"][b, 0], (extra, b)


def test_config3_motion_track_60s_int16_from_rinex(tmp_path):
    """BASELINE configs[3] (motion file, --iq16, 60 s = 599 blocks, 718.8 MB): scenario engine +
    CUDA synthesis against the reference's stream for the same generated track."""
    import motion_track
    g = scenario.load_golden("sky12_track_60s_i16")
    mot = tmp_path / "track.csv"
    motion_track.write_motion(str(mot), 600)
    ch, nav = gps.scenario(_nav_file(tmp_path, 12), 35.681298, 139.766247, 10.0, seconds=60, max_chan=12,
                           motion_file=str(mot), start=(2024, 1, 7, 2, 0, 0.0))
    assert ch.shape == (599, 12)
    with gps.Context(12, 599, max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 2)
    assert np.array_equal(scenario.crc_blocks(out), g["crcs"][:, 0])


def test_device_carrier_chain_equals_sequential_host_chain():
    ch, nav = gps.synthetic_chans(130, 32, seed=21)
    with gps.Context(32, 50) as ctx:                      # 130 blocks > max_blocks: windows of 50
        got = ctx.carrier_chain(ch)
        assert np.array_equal(got, gps.carrier_chain(ch, threads=4))
        mid = ctx.carrier_chain(ch[:70])
        assert np.array_equal(ctx.carrier_chain(ch[70:], phase_in=mid), got)


def test_channel_reallocation_and_gaps_vs_oracle():
    # slots that change satellite, go idle and come back inside one call (allocateChannel every 30 s, gps.c:2909)
    ch, nav = gps.synthetic_chans(6, 12, seed=33)
    ch["prn"][2:, 3] = 0                                   # slot 3 drops out after two blocks
    ch["prn"][3:, 5] = 31                                  # slot 5 switches satellite at block 3
    ch["carr_phase"][3, 5] = 0.6180339887
    ch["prn"][1:3, 7] = 0                                  # slot 7 pauses for two blocks, then resumes
    ch["carr_phase"][3, 7] = 0.25
    for ss in (1, 2):
        want, carr = scenario.oracle_run(ch, nav, ss)
        with gps.Context(12, 6) as ctx:
            ctx.set_nav_frames(nav)
            out, cp = ctx.synth_blocks(ch, ss)
        assert np.array_equal(out, want)
        assert np.array_equal(cp, carr)


@pytest.mark.parametrize("knob,val", [("GPSB200_GRADED_CHUNKS", "0")])
def test_experiment_knobs_do_not_change_the_output(knob, val, monkeypatch):
    # the knobs of README.md only move work around (download chunking)
    ch, nav = gps.synthetic_chans(300, 32, seed=4242)
    with gps.Context(32, 300) as ctx:
        ctx.set_nav_frames(nav)
        want, cp = ctx.synth_blocks(ch, 1)
    monkeypatch.setenv(knob, val)
    with gps.Context(32, 300) as ctx:
        ctx.set_nav_frames(nav)
        got, cp2 = ctx.synth_blocks(ch, 1)
    assert np.array_equal(got, want) and np.array_equal(cp, cp2)


def test_two_contexts_used_concurrently_from_two_threads():
    import threading
    cases = [gps.synthetic_chans(40, 32, seed=901), gps.synthetic_chans(40, 12, seed=902)]
    want = []
    for ch, nav in cases:
        with gps.Context(ch.shape[1], 40) as ctx:
            ctx.set_nav_frames(nav)
            want.append(ctx.synth_blocks(ch, 1)[0])
    got = [None, None]

    def work(k):
        ch, nav = cases[k]
        with gps.Context(ch.shape[1], 40) as ctx:
            ctx.set_nav_frames(nav)
            for _ in range(3):
                got[k] = ctx.synth_blocks(ch, 1)[0]

    th = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for k in range(2):
        assert np.array_equal(got[k], want[k]), k


def test_single_block_call_latency_is_far_below_real_time():
    # the reference's cadence: one 0.1 s block per call (INTEGRATION.md section 1)
    import time
    ch, nav = gps.synthetic_chans(20, 12, seed=8)
    with gps.Context(12, 1) as ctx:
        ctx.set_nav_frames(nav)
        cp = None
        out = np.empty(gps.BLOCK_ELEMS, np.int8)
        times = []
        for b in range(20):
            one = ch[b:b + 1].copy()
            if cp is not None:
                one["carr_phase"][0] = cp
            t0 = time.perf_counter()
            _, cp = ctx.synth_blocks(one, 1, out=out)
            times.append(time.perf_counter() - t0)
    med = sorted(times[3:])[len(times[3:]) // 2]
    print("single-block call: median %.2f ms" % (med * 1e3))
    assert med < 0.05                                      # a block is 100 ms of signal


def test_chain_self_check_catches_corruption():
    # defence in depth: k_checkpoints re-derives every block's end phase by an exact walk and compares it
    # with the start phase the two-level speculation resolved for the next block; a corruption by one unit of
    # the rounding grid (gpsb200_debug_corrupt_chain) must be reported. The hook corrupts the first span of slot 0:
    # a regular span, resolved from its span summary, and -- slot 0 changes satellite at block 3 -- a span the host
    # resolved block by block
    import torch
    for realloc in (False, True):
        ch, nav = gps.synthetic_chans(12, 32, seed=77)
        if realloc:
            ch["prn"][3:, 0] = ch["prn"][0, 0] % 32 + 1
            ch["carr_phase"][3, 0] = 0.25
        with gps.Context(32, 12) as ctx:
            ctx.set_nav_frames(nav)
            good, _ = ctx.synth_blocks(ch, 1)
            ctx.debug_corrupt_chain(True)
            with pytest.raises(gps.GpsB200Error) as e:
                ctx.synth_blocks(ch, 1)
            assert e.value.code == -5, realloc
            # the device-destination path reports it as well, with or without a stats request
            dev = torch.empty(12 * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
            with pytest.raises(gps.GpsB200Error) as e:
                ctx.synth_blocks_device(ch, 1, dev.data_ptr())
            assert e.value.code == -5, realloc
            # ... and so does the three-step slice call, at gpsb200_slice_wait
            ctx.slice_prepare(ch, 1, dev.data_ptr())
            ctx.slice_probe()
            ctx.slice_finish()
            with pytest.raises(gps.GpsB200Error) as e:
                ctx.slice_wait()
            assert e.value.code == -5, realloc
            ctx.debug_corrupt_chain(False)
            again, _ = ctx.synth_blocks(ch, 1)
            assert np.array_equal(good, again)


def test_full_size_3600s_32ch_device_path_properties():
    """BASELINE configs[4] at full size on ONE GPU (35 999 blocks x 32 channels = 10.8 Gsamples, 21.6 GB in
    HBM): the parallel-in-time chain over a whole hour equals the sequential exact chain, and sampled
    blocks equal the CPU oracle started from sequentially computed phases."""
    import torch
    nblk, nchan = 35999, 32
    ch, nav = gps.synthetic_chans(nblk, nchan, seed=2024)
    with gps.Context(nchan, nblk) as ctx:
        ctx.set_nav_frames(nav)
        dev = torch.empty(nblk * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
        cp, st = ctx.synth_blocks_device(ch, 1, dev.data_ptr(), want_stats=True)
        torch.cuda.synchronize()
        assert st.chain_fallbacks < 0.01 * nblk * nchan
        assert np.array_equal(cp, gps.carrier_chain(ch, threads=16))
        for b in (20000, 35998):
            start = ctx.carrier_chain(ch[:b])                 # device chain of the prefix ...
            assert np.array_equal(start, gps.carrier_chain(ch[:b], threads=16))   # ... equals the host one
            one = ch[b:b + 1].copy()
            one["carr_phase"][0] = start
            want, _ = scenario.oracle_run(one, nav, 1)
            got = dev[b * gps.BLOCK_ELEMS:(b + 1) * gps.BLOCK_ELEMS].cpu().numpy()
            assert np.array_equal(got, want), b


def test_randomized_differential_vs_oracle():
    """Seeded differential test: 40 one-block cases with parameters drawn far beyond what a real
    constellation produces (Doppler to +-30 kHz, tiny gains, code phases and NAV positions at their
    edges, word/bit roll-over inside the block, several NAV frames, unused slots, int8 and int16)."""
    rng = np.random.default_rng(20240107)
    for case in range(40):
        nchan = int(rng.choice([1, 3, 8, 12, 16, 20, 32]))
        ss = int(rng.choice([1, 2]))
        nblk = int(rng.choice([1, 2, 3, 4]))             # 1-2: host-resolved small-call path, 3+: speculative chain
        ch, _ = gps.synthetic_chans(nblk, nchan, seed=1000 + case)
        nframes = 3
        nav = rng.integers(0, 1 << 32, size=(nframes, nchan, 60), dtype=np.uint32)   # incl. garbage in bits 30..31
        ch["nav_frame"] = rng.integers(0, nframes, size=(nblk, 1))
        scale = rng.choice([1.0, 6.0, 0.01, 1e-5])
        ch["f_carr"] *= scale
        ch["f_code"] = 1.023e6 + ch["f_carr"] / 1540.0
        ch["gain"] = rng.uniform(0.0, 1.2, size=ch["gain"].shape) * rng.choice([1.0, 0.02])
        edge = rng.integers(0, 4, size=nchan)
        ch["code_phase"][:, edge == 1] = np.nextafter(1023.0, 0)
        ch["code_phase"][:, edge == 2] = 0.0
        ch["icode"][:, edge == 3] = 19
        ch["ibit"][:, edge == 3] = 29                                              # word roll-over inside the block
        ch["iword"][:, edge == 3] = rng.integers(0, 59)
        ch["carr_phase"][0] = rng.choice([0.0, np.nextafter(1.0, 0), 0.5, 2.0 ** -40], size=nchan)
        ch["prn"][:, rng.random(nchan) < 0.15] = 0
        want, carr = scenario.oracle_run(ch, nav, ss)
        with gps.Context(nchan, nblk, max_nav_frames=nframes) as ctx:
            ctx.set_nav_frames(nav)
            out, cp = ctx.synth_blocks(ch, ss)
        assert np.array_equal(out, want), (case, nchan, ss, scale)
        assert np.array_equal(cp, carr), case


def test_config3_literally_circle_csv_int16_60s_from_rinex(tmp_path):
    """BASELINE configs[3] LITERALLY: the reference's own circle.csv (rows carried in the fixture, re-written with
    %.17g so that every double parses back identically), --iq16, 60 s = 599 blocks: RINEX + motion file in,
    the reference's int16 stream out."""
    g = scenario.load_golden("sky12_circle_60s_i16")
    mot = tmp_path / "circle.csv"
    with open(mot, "w") as f:
        for r in g["motion_rows"]:
            f.write("%.17g,%.17g,%.17g,%.17g\n" % tuple(r))
    ch, nav = gps.scenario(_nav_file(tmp_path, 12), 35.681298, 139.766247, 10.0, seconds=60, max_chan=12,
                           motion_file=str(mot), start=(2024, 1, 7, 2, 0, 0.0))
    assert ch.shape == (599, 12)
    for f in ("prn", "f_carr", "f_code", "code_phase", "gain", "iword", "ibit", "icode"):     # first two blocks: dumped
        assert np.array_equal(ch[f][:2], g["chans"][f]), f
    with gps.Context(12, 599, max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 2)
    bad = np.nonzero(scenario.crc_blocks(out) != g["crcs"][:, 0])[0]
    assert bad.size == 0, bad[:10]


def test_pluto_gain_int16_matches_reference_stream(tmp_path):
    """ADALM-Pluto flavour of the loop: gain x 2 (gps.c:2759-2763), int16 (sdr_pluto.c:107-110). Once from the
    reference's dumped parameters, once from the RINEX file through the scenario engine (pluto_gain=True)."""
    g, out = run_golden("sky12_pluto_3s_i16")
    assert np.array_equal(out[:gps.BLOCK_ELEMS], g["keep_blocks"][0])
    ch, nav = gps.scenario(_nav_file(tmp_path, 12), 35.681298, 139.766247, 10.0, seconds=3, max_chan=12,
                           start=(2024, 1, 7, 2, 0, 0.0), pluto_gain=True)
    assert np.array_equal(ch["gain"], g["chans"]["gain"])
    with gps.Context(12, ch.shape[0], max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out2, _ = ctx.synth_blocks(ch, 2)
    assert np.array_equal(scenario.crc_blocks(out2), g["crcs"][:, 0])


def test_rinex3_file_to_reference_stream(tmp_path):
    """RINEX-3 navigation file (readRinex3, gps.c:1512-1891) -> scenario engine -> CUDA synthesis == the reference's
    stream for the same file read with -3."""
    import os
    import subprocess
    import sys
    g = scenario.load_golden("sky12_rinex3_3s_i8")
    nav_file = tmp_path / "sky12.rnx"
    subprocess.check_call([sys.executable, os.path.join(scenario.ROOT, "oracle", "gen_rinex.py"), "--nsat", "12", "--v3",
                           "--out", str(nav_file)])
    ch, nav = gps.scenario(str(nav_file), 35.681298, 139.766247, 10.0, seconds=3, max_chan=12,
                           start=(2024, 1, 7, 2, 0, 0.0), rinex3=True)
    with gps.Context(12, ch.shape[0], max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 1)
    assert np.array_equal(scenario.crc_blocks(out), g["crcs"][:, 0])


def _sliced_stream_crcs(ch, nav, edges, sample_size=1):
    """Synthesize one scenario as len(edges)-1 time slices, each by its own context ("rank"), sequentially on
    this device: a rank knows only the parameters and the exact carrier phases handed over by the chain through the
    blocks before its slice (sharding.start_phases / seed_slice) -- never another rank's output."""
    crcs = []
    nchan = ch.shape[1]
    for lo, hi in zip(edges[:-1], edges[1:]):
        with gps.Context(nchan, hi - lo, max_nav_frames=len(nav)) as ctx:
            ctx.set_nav_frames(nav)
            part = ch[lo:hi]
            if lo > 0:
                part = gps.sharding.seed_slice(part, ch[lo - 1], gps.sharding.start_phases(ch[:lo], ctx=ctx))
            out, _ = ctx.synth_blocks(part, sample_size)
            crcs.append(scenario.crc_blocks(out))
    return np.concatenate(crcs)


@pytest.mark.parametrize("ranks", [2, 4, 8])
def test_time_sliced_stream_equals_reference_stream(ranks, tmp_path):
    """SURVEY section 8e on one device: the 310 s / 32-channel reallocation scenario cut into K slices, every slice
    made by a separate context from the hand-over phases alone; the concatenation is the reference's stream. One
    extra cut is placed exactly on the block where a satellite rises into a free slot (block 2399/2400: the slot
    must take its allocation phase, not a chained one) and one where a satellite sets."""
    g = scenario.load_golden("sky32_lat60_310s_i8")
    ch, nav = gps.scenario(_nav_file(tmp_path, 32), 60.0, 140.0, 0.0, seconds=310, max_chan=32, start=(2024, 1, 7, 2, 0, 0.0))
    occ = ch["prn"]
    change = [b for b in range(1, ch.shape[0]) if np.any(occ[b] != occ[b - 1])]
    assert change, "the scenario is expected to reallocate"
    edges = sorted(set([gps.sharding.slice_bounds(ch.shape[0], ranks, r)[0] for r in range(ranks)] + change + [ch.shape[0]]))
    got = _sliced_stream_crcs(ch, nav, edges)
    bad = np.nonzero(got != g["crcs"][:, 0])[0]
    assert bad.size == 0, (edges, bad[:10])


def _three_step_slices(ch, nav, edges, sample_size=1):
    """The hand-over protocol of include/gpsb200.h on one device: every slice gets its own context ("rank");
    all ranks first run gpsb200_slice_prepare (links), the links are composed into GUESSED incoming states, every
    rank probes speculatively from its guess, and only then the exact states travel rank to rank through
    gpsb200_slice_finish. -> (block CRCs of the concatenated stream, total sequential fallbacks)"""
    import torch
    nchan = ch.shape[1]
    ctxs, outs, links = [], [], []
    try:
        for lo, hi in zip(edges[:-1], edges[1:]):
            ctx = gps.Context(nchan, hi - lo, max_nav_frames=len(nav))
            ctx.set_nav_frames(nav)
            dev = torch.empty((hi - lo) * gps.BLOCK_ELEMS, dtype=torch.int8 if sample_size == 1 else torch.int16,
                              device="cuda")
            ctxs.append(ctx)
            outs.append(dev)
            links.append(ctx.slice_prepare(ch[lo:hi], sample_size, dev.data_ptr()))
        prn, ph = None, None
        for k, (ctx, link) in enumerate(zip(ctxs, links)):    # guesses: closed form only, no GPU result involved
            ctx.slice_probe(prn, ph, eager=k + 1 < len(ctxs))
            prn, ph = gps.link_apply(link, nchan, prn, ph)
        prn, ph, fallbacks = None, None, 0
        for ctx in ctxs:                                      # exact states, rank to rank
            handed = []
            prn, ph, st = ctx.slice_finish(prn, ph, want_stats=True, handoff=lambda a, b: handed.append((a, b)))
            assert len(handed) == 1 and np.array_equal(handed[0][0], prn) and np.array_equal(handed[0][1], ph)
            fallbacks += st.chain_fallbacks
        for ctx in ctxs:
            ctx.slice_wait()                                  # completion + verdict of the device self-check
        torch.cuda.synchronize()
        crcs = np.concatenate([scenario.crc_blocks(o.cpu().numpy()) for o in outs])
        return crcs, fallbacks, (prn, ph)
    finally:
        for ctx in ctxs:
            ctx.close()


@pytest.mark.parametrize("ranks", [2, 8])
def test_three_step_hand_over_equals_reference_stream(ranks, tmp_path):
    """gpsb200_slice_prepare / _probe / _finish over K "ranks" of the 310 s reallocation scenario (cuts also on the
    blocks where a satellite rises or sets): the concatenation is the reference's stream, and the exact state after
    the last slice equals the one-call result."""
    g = scenario.load_golden("sky32_lat60_310s_i8")
    ch, nav = gps.scenario(_nav_file(tmp_path, 32), 60.0, 140.0, 0.0, seconds=310, max_chan=32, start=(2024, 1, 7, 2, 0, 0.0))
    occ = ch["prn"]
    change = [b for b in range(1, ch.shape[0]) if np.any(occ[b] != occ[b - 1])]
    edges = sorted(set([gps.sharding.slice_bounds(ch.shape[0], ranks, r)[0] for r in range(ranks)] + change + [ch.shape[0]]))
    got, fallbacks, (prn, ph) = _three_step_slices(ch, nav, edges)
    bad = np.nonzero(got != g["crcs"][:, 0])[0]
    assert bad.size == 0, (edges, bad[:10])
    assert fallbacks < 0.01 * ch.size
    want = gps.carrier_chain(ch, threads=8)
    assert np.array_equal(ph, want)
    assert np.array_equal(prn, np.where(occ[-1] > 0, occ[-1], 0))


def test_reference_program_with_the_drop_in_patch_writes_the_reference_stream(tmp_path):
    """INTEGRATION.md section 1 compiled and run: oracle/_ref/ref_gpsb200_12 is the reference program -- its own
    producer thread with the 10 Hz path, NAV generation and channel allocation (gps.c), its own sink dispatch and
    iqfile writer (sdr.c, sdr_iqfile.c), all unmodified -- with ONLY the sample loop + quantise/pack (gps.c:2767-2857)
    replaced by gpsb200_synth_blocks (oracle/ref_harness/apply_integration.py, integration_*.inc) and libgpsb200.so
    linked instead of fifo.o. BASELINE configs[1]: the iqdata.bin it writes equals the reference's enqueue stream,
    all 99 blocks (our FIFO does not drop buffers 1..6)."""
    import os
    import subprocess
    import zlib
    exe = os.path.join(scenario.ROOT, "oracle", "_ref", "ref_gpsb200_12")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_gpsb200_12 not built (needs the reference sources)")
    nav = _nav_file(tmp_path, 12)
    g = scenario.load_golden("sky12_static_10s_i8")
    r = subprocess.run([exe, "-e", nav, "-l", "35.681298,139.766247,10.0", "-d", "10"], cwd=tmp_path,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-600:]
    s = np.fromfile(tmp_path / "iqdata.bin", dtype=np.int8)
    assert s.size == 99 * gps.BLOCK_ELEMS, s.size
    for b, row in enumerate(s.reshape(99, gps.BLOCK_ELEMS)):
        assert zlib.crc32(row.tobytes()) == g["crcs"][b, 0], b


def test_config4_3600s_32ch_sliced_8_ways_equals_reference_stream(tmp_path):
    """BASELINE configs[4] LITERALLY: 32 channels, int8, 3600 s = 35 999 blocks = 10.8 Gsamples, time-sliced 8 ways
    (the three-step hand-over, every slice by its own context), RINEX file in -- against the CRC-32 of every block of
    the reference's own 3600 s run (tests/golden/sky32_static_3600s_i8.npz; 35 minutes of one CPU for the reference).
    The scenario includes satellites setting and slots being reallocated during the hour."""
    import torch
    g = scenario.load_golden("sky32_static_3600s_i8")
    ch, nav = gps.scenario(_nav_file(tmp_path, 32), 35.681298, 139.766247, 10.0, seconds=3600, max_chan=32,
                           start=(2024, 1, 7, 2, 0, 0.0))
    assert ch.shape == (35999, 32)
    ranks = 8
    edges = [gps.sharding.slice_bounds(ch.shape[0], ranks, r)[0] for r in range(ranks)] + [ch.shape[0]]
    nchan = 32
    ctxs, links = [], []
    dev = torch.empty(max(b - a for a, b in zip(edges[:-1], edges[1:])) * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
    bad_total = 0
    try:
        # links first (closed form), composed into guessed incoming states
        guesses = []
        prn, ph = None, None
        for lo, hi in zip(edges[:-1], edges[1:]):
            guesses.append((prn, ph))
            prn, ph = gps.link_apply(gps.slice_link_host(ch[lo:hi]), nchan, prn, ph)
        eprn, eph = None, None
        for (lo, hi), (gprn, gph) in zip(zip(edges[:-1], edges[1:]), guesses):
            with gps.Context(nchan, hi - lo, max_nav_frames=len(nav)) as ctx:      # one "rank" at a time: 2.7 GB each
                ctx.set_nav_frames(nav)
                ctx.slice_prepare(ch[lo:hi], 1, dev.data_ptr())
                ctx.slice_probe(gprn, gph, eager=hi < ch.shape[0])
                eprn, eph, st = ctx.slice_finish(eprn, eph, want_stats=True)
                ctx.slice_wait()
                assert st.chain_fallbacks < 0.01 * (hi - lo) * nchan
                got = scenario.crc_blocks(dev[:(hi - lo) * gps.BLOCK_ELEMS].cpu().numpy())
            bad = np.nonzero(got != g["crcs"][lo:hi])[0]
            bad_total += bad.size
            assert bad.size == 0, (lo, hi, bad[:10] + lo)
    finally:
        for c in ctxs:
            c.close()
    assert bad_total == 0
    assert np.array_equal(eph, gps.carrier_chain(ch, threads=16))


def test_target_option_static_start_point_matches_reference_stream(tmp_path):
    """-t distance,bearing,height (gps-sim.c:145-148, gps.c:2348-2357): scenario engine + synthesis against the
    reference run with the same option."""
    g = scenario.load_golden("sky12_target_3s_i8")
    ch, nav = gps.scenario(_nav_file(tmp_path, 12), 35.681298, 139.766247, 10.0, seconds=3, max_chan=12,
                           start=(2024, 1, 7, 2, 0, 0.0), target=(1500.5, 33.3, 120.25))
    with gps.Context(12, ch.shape[0], max_nav_frames=len(nav)) as ctx:
        ctx.set_nav_frames(nav)
        out, _ = ctx.synth_blocks(ch, 1)
    assert np.array_equal(scenario.crc_blocks(out), g["crcs"][:, 0])


def test_cli_multi_gpu_slices_write_the_reference_stream(tmp_path):
    """gpsb200-sim --gpus N (one worker thread + context per device, slices handed over with the three-step API, one
    FIFO sink in stream order) and the zero-copy single-GPU path with -t: CRC-equal to the reference goldens.
    N = 2 when two devices are visible, else the N = 1 paths only."""
    import os
    import subprocess
    import zlib
    import torch
    exe = os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "gpsb200-sim")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "csrc")])
    nav = _nav_file(tmp_path, 12)
    base = [exe, "-e", nav, "-l", "35.681298,139.766247,10.0", "-s", "2024/01/07,02:00:00"]
    g = scenario.load_golden("sky12_static_35s_i8")
    counts = [1] + ([2] if torch.cuda.device_count() >= 2 else [])
    for n in counts:
        out = tmp_path / ("iq_%d.bin" % n)
        subprocess.check_call(base + ["-d", "35", "--gpus", str(n), "-o", str(out)])
        s = np.fromfile(out, dtype=np.int8).reshape(-1, gps.BLOCK_ELEMS)
        assert s.shape[0] == 349
        bad = [b for b, row in enumerate(s) if zlib.crc32(row.tobytes()) != g["crcs"][b, 0]]
        assert not bad, (n, bad[:5])
    gt = scenario.load_golden("sky12_target_3s_i8")
    out = tmp_path / "iq_t.bin"
    subprocess.check_call(base + ["-d", "3", "-t", "1500.5,33.3,120.25", "-o", str(out)])
    s = np.fromfile(out, dtype=np.int8).reshape(-1, gps.BLOCK_ELEMS)
    assert [zlib.crc32(r.tobytes()) for r in s] == list(gt["crcs"][:, 0])


def test_fewer_channels_than_the_context_was_created_for():
    """nchan <= cfg.max_chan: a 32-slot context synthesizing 12-channel calls (NAV rows are indexed by the context's
    slots) equals a 12-slot context."""
    ch, nav = gps.synthetic_chans(5, 12, seed=515)
    with gps.Context(12, 5) as ctx:
        ctx.set_nav_frames(nav)
        want, cp = ctx.synth_blocks(ch, 1)
    with gps.Context(32, 8) as ctx:
        ctx.set_nav_frames(nav)
        got, cp2 = ctx.synth_blocks(ch, 1)
    assert np.array_equal(got, want) and np.array_equal(cp, cp2)


@pytest.mark.parametrize("nchan,ss", [(1, 1), (5, 2), (8, 1), (12, 1), (12, 2), (16, 2), (17, 1), (23, 2), (32, 1), (32, 2)])
def test_both_synthesis_kernels(nchan, ss, monkeypatch):
    """k_synth_lanes (lane = sample; the 16- and the 32-channel variant) is the default; GPSB200_LANES=0 keeps calls on
    k_synth's 8-, 16- and 32-lane variants. Both against the oracle, 5 blocks (speculative chain path), odd window count
    per run and odd channel counts included."""
    ch, nav = scenario.synthetic_chans(5, nchan, seed=700 + nchan)
    ch["prn"][:, nchan // 2] = 0 if nchan > 4 else ch["prn"][:, nchan // 2]            # an idle slot in the middle
    want, carr = scenario.oracle_run(ch, nav, ss)
    for lanes_on, name in (("1", "k_synth_lanes"), ("0", "k_synth")):
        monkeypatch.setenv("GPSB200_LANES", lanes_on)
        with gps.Context(nchan, 5) as ctx:
            ctx.set_nav_frames(nav)
            out, cp = ctx.synth_blocks(ch, ss)
            assert ctx.synth_kernel_name(nchan) == name
        assert np.array_equal(out, want), name
        assert np.array_equal(cp, carr), name


def test_lanes_kernel_declines_code_rates_outside_its_range():
    """f_code far from 1.023 MHz (legal for the API: <= 1.07 MHz) keeps the context on k_synth; output still exact."""
    ch, nav = scenario.synthetic_chans(3, 8, seed=811)
    ch["f_code"][:, 3] = 1.06e6
    want, carr = scenario.oracle_run(ch, nav, 1)
    with gps.Context(8, 3) as ctx:
        ctx.set_nav_frames(nav)
        assert ctx.synth_kernel_name(8) == "k_synth_lanes"
        out, cp = ctx.synth_blocks(ch, 1)
        assert ctx.synth_kernel_name(8) == "k_synth"
    assert np.array_equal(out, want) and np.array_equal(cp, carr)
