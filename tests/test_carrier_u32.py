"""The reference's INTEGER carrier NCO build (gps.h:17 without `#define FLOAT_CARR_PHASE`): unsigned 32-bit carr_phase,
carr_phasestep = (int) round(512.0 * 65536.0 * f_carr * delt) per block, index (carr_phase >> 16) & 511, modulo-2^32
add per sample (gps.c:2745-2747, 2777, 2828). A GPSB200_CARRIER_U32 context reproduces that stream bit for bit.

CPU: the oracle of that build against the reference's own stream (tests/golden/*_u32.npz, make_golden_u32.py), the
scenario engine's allocation phases, the host model of the lane = sample kernel, the exact slice links.
GPU: every U32 golden stream through every path of the library, both synthesis kernels, the CLI, the drop-in program."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib
import refdump
import scenario
from scenario import gps

LOC = (35.681298, 139.766247, 10.0)
LOC60 = (60.0, 140.0, 0.0)
START = (2024, 1, 7, 2, 0, 0.0)
CIRCLE = os.path.join(scenario.GOLD, "circle.csv")
TWO32 = 1 << 32

# ---- the oracle of the integer build (oracle/gpsl1_oracle_u32.c) ------------------------------------------------------
_SO = os.path.join(scenario.ROOT, "oracle", "_ref", "liboracle_gpsl1_u32.so")
_olib = None


def olib():
    global _olib
    if _olib is None:
        if not os.path.exists(_SO):
            subprocess.check_call(["make", "-C", os.path.join(scenario.ROOT, "oracle"), "-f", "u32.mk",
                                   "_ref/liboracle_gpsl1_u32.so"])
        _olib = C.CDLL(_SO)
        _olib.oracle_synth_block_u32.argtypes = [C.POINTER(oracle_lib.OracleChan), C.c_int, C.c_int, C.c_void_p]
    return _olib


def oracle_block_u32(row, nav_row, carr):
    chans = oracle_lib.make_chans(row, nav_row, carr)
    iq = np.zeros(2 * gps.BLOCK_SAMPLES, np.int16)
    olib().oracle_synth_block_u32(chans, len(chans), gps.BLOCK_SAMPLES, iq.ctypes.data)
    return iq, np.array([c.carr_phase if c.prn > 0 else 0.0 for c in chans])


def oracle_run_u32(ch, nav, sample_size):
    """The oracle over chans[nblk, C], chaining the u32 phase like the library (a slot's first block, or a new satellite
    in it, takes carr_phase)."""
    nblk, nchan = ch.shape
    outs, carr, prev = [], np.zeros(nchan), np.zeros(nchan, np.int32)
    for b in range(nblk):
        row = ch[b]
        cp = np.where((row["prn"] == prev) & (b > 0), carr, row["carr_phase"])
        iq, carr = oracle_block_u32(row, nav[int(row["nav_frame"][0])], cp)
        outs.append(iq if sample_size == 2 else oracle_lib.quantize8(iq))
        prev = row["prn"].copy()
    return np.concatenate(outs), carr


def u32_synthetic(nblk, nchan, seed, **kw):
    """synthetic_chans with u32 start phases."""
    ch, nav = gps.synthetic_chans(nblk, nchan, seed=seed, **kw)
    rng = np.random.default_rng(seed + 12345)
    ch["carr_phase"] = 0.0
    ch["carr_phase"][0] = rng.integers(0, TWO32, nchan).astype(np.float64)
    return ch, nav


def make_nav(tmp_path, nsat):
    nav = tmp_path / ("sky%d.nav" % nsat)
    subprocess.check_call([sys.executable, os.path.join(scenario.ROOT, "oracle", "gen_rinex.py"),
                           "--nsat", str(nsat), "--out", str(nav)])
    return str(nav)


def event_edges(ch, ranks):
    """Slice edges of ch: K near-equal slices plus a cut on every block where a slot's satellite changes."""
    occ = ch["prn"]
    change = [b for b in range(1, ch.shape[0]) if np.any(occ[b] != occ[b - 1])]
    assert change, "the scenario is expected to reallocate"
    even = [gps.sharding.slice_bounds(ch.shape[0], ranks, r)[0] for r in range(ranks)]
    return sorted(set(even + change + [ch.shape[0]]))


# ======================================================================================================================
# CPU
# ======================================================================================================================
@pytest.mark.parametrize("name", ["sky12_static_10s_i8_u32", "sky32_static_10s_i8_u32", "sky12_circle_60s_i16_u32",
                                  "sky32_lat60_310s_i8_u32"])
def test_oracle_u32_reproduces_the_integer_reference_stream(name):
    """oracle_synth_block_u32 from the dumped parameters (carr_phase = the dumped u32 phase at block start): every block
    whose parameters the fixture holds has the reference's CRCs (whole block and its 30 parts); kept blocks verbatim."""
    g = scenario.load_golden(name)
    ch, frames = scenario.golden_chans(g)
    idx = g["chans_idx"] if "chans_idx" in g.files else np.arange(ch.shape[0])
    ss = int(g["sample_size"])
    keep = dict(zip(g["keep_idx"].tolist(), g["keep_blocks"]))
    fidx = g["nav_frame_of_block"]                       # indexed by block number (chans may hold a subset)
    for j, b in enumerate(idx):
        iq, _ = oracle_block_u32(ch[j], frames[int(fidx[b])], None)
        out = iq if ss == 2 else oracle_lib.quantize8(iq)
        assert np.array_equal(refdump.block_crcs(out)[0], g["crcs"][b]), (name, int(b))     # whole block + 30 parts
        if int(b) in keep:
            assert np.array_equal(out, keep[int(b)])


def test_dumped_u32_phases_follow_the_closed_form():
    """The fixture's own block-start phases: u[b+1] = u[b] + 300000 * step[b] mod 2^32 while the slot keeps its
    satellite (the closed form the library uses instead of a carrier chain)."""
    for name in ("sky12_static_10s_i8_u32", "sky32_static_10s_i8_u32", "sky12_circle_60s_i16_u32"):
        ch, _ = scenario.golden_chans(scenario.load_golden(name))
        for b in range(ch.shape[0] - 1):
            for c in np.nonzero((ch["prn"][b] > 0) & (ch["prn"][b] == ch["prn"][b + 1]))[0]:
                want = gps.carrier_advance_u32(ch["carr_phase"][b, c], ch["f_carr"][b, c], gps.BLOCK_SAMPLES)
                assert ch["carr_phase"][b + 1, c] == want, (name, b, c)


@pytest.mark.parametrize("name,nsat,secs,loc", [("sky12_static_10s_i8_u32", 12, 10, LOC),
                                                ("sky32_lat60_310s_i8_u32", 32, 310, LOC60)])
def test_scenario_engine_u32_matches_the_integer_reference_dump(name, nsat, secs, loc, tmp_path):
    """carrier='u32': the allocation phases are the reference's (unsigned int) (512 * 65536 * frac(phase_ini))
    (gps.c:2212-2213), bit for bit; every other record is the FP64 engine's, which equals the integer build's dump."""
    g = scenario.load_golden(name)
    want, _ = scenario.golden_chans(g)
    idx = g["chans_idx"] if "chans_idx" in g.files else np.arange(want.shape[0])
    nav_file = make_nav(tmp_path, nsat)
    got, nav = gps.scenario(nav_file, *loc, seconds=secs, max_chan=nsat, start=START, carrier="u32")
    f64, nav64 = gps.scenario(nav_file, *loc, seconds=secs, max_chan=nsat, start=START)
    for f in gps.CHAN_DTYPE.names:
        if f != "carr_phase":
            assert np.array_equal(got[f], f64[f]), f
    assert np.array_equal(nav, nav64)
    act = got["prn"] > 0
    u = got["carr_phase"][act]
    assert np.all((u >= 0) & (u < TWO32) & (u == np.floor(u)))
    assert np.array_equal(got["carr_phase"][act], np.floor(f64["carr_phase"][act] * 33554432.0))
    sub = got[idx]
    assert np.array_equal(sub["prn"], want["prn"])
    a = want["prn"] > 0
    for f in ("iword", "ibit", "icode", "f_carr", "f_code", "code_phase", "gain"):
        assert np.array_equal(sub[f][a], want[f][a]), f
    # allocation phases: block 0, and every block where a slot takes a new satellite
    prev = np.zeros(got.shape[1], np.int32)
    alloc = np.zeros(got.shape, bool)
    for b in range(got.shape[0]):
        alloc[b] = (got["prn"][b] > 0) & (got["prn"][b] != prev)
        prev = got["prn"][b]
    fresh = alloc[idx] & a
    assert fresh[0].any()
    assert np.array_equal(sub["carr_phase"][fresh], want["carr_phase"][fresh])
    if "prn_of_block" in g.files:
        assert np.array_equal(got["prn"].astype(np.int8), g["prn_of_block"])


def _lanes_case(nchan, seed):
    ch, nav = u32_synthetic(1, nchan, seed)
    rng = np.random.default_rng(seed)
    row = ch[0]
    # edge cases spread over the slots: a phase just below 2^32, zero / negative / largest steps, a code phase right
    # before a code-period boundary in the last period of a NAV bit (a NAV bit change inside the first samples)
    row["carr_phase"][0] = TWO32 - 1 - int(rng.integers(0, 5000))
    if nchan > 1:
        row["f_carr"][1] = 0.0
    if nchan > 2:
        row["f_carr"][2] = -2.899e6
    if nchan > 3:
        row["f_carr"][3] = 2.899e6
        row["carr_phase"][3] = TWO32 - 1
    if nchan > 4:
        row["f_carr"][4] = -1.0 / 3.0
    for c in range(5, nchan, 3):
        row["code_phase"][c] = 1023.0 - rng.uniform(0, 5)
        row["icode"][c] = 19
    return ch, nav


@pytest.mark.parametrize("nchan", [1, 2, 5, 12, 16, 17, 29, 32])
@pytest.mark.parametrize("run_samples", [96, 480, 2400])
def test_lanes_model_u32_equals_oracle(nchan, run_samples):
    """The lane = sample algorithm in U32 mode (host model of k_synth_lanes<.., U32>) against the oracle of the integer
    build: phases crossing 2^32, zero / negative / largest steps, NAV bit changes at code-period boundaries, every run
    length the kernel accepts (multiples of 96 dividing 300000, up to 2400)."""
    ch, nav = _lanes_case(nchan, seed=900 + nchan + run_samples)
    want, carr = oracle_block_u32(ch[0], nav[0], None)
    iq, co, cnt = gps.lanes_model_block(ch[0], nav[0], run_samples=run_samples, carrier="u32")
    assert np.array_equal(iq, want)
    assert np.array_equal(co, carr)
    assert cnt[1] == 0 and cnt[3] == 0                     # the u32 index never needs a repair


def test_lanes_model_u32_rejects_non_integer_phases():
    ch, nav = u32_synthetic(1, 4, seed=3)
    ch["carr_phase"][0, 1] = 0.5
    with pytest.raises(gps.GpsB200Error):
        gps.lanes_model_block(ch[0], nav[0], carrier="u32")


def test_u32_step_matches_the_reference_evaluation():
    """carrier_advance_u32's step is (int) round((33554432.0 * f) * delt) with C rounding (ties away from zero)."""
    assert gps.carrier_advance_u32(0, 0.0, 1) == 0.0
    assert gps.carrier_advance_u32(5, -1.0 / 3.0, 1) == 1.0              # -3.73 rounds to -4
    assert gps.carrier_advance_u32(0, -3000000.0 / 33554432.0 * 0.5, 1) == float(TWO32 - 1)   # -0.5: away from zero
    for f in (1234.5, -4321.25, 2.899e6, -2.899e6, 0.1):
        x = (33554432.0 * f) * (1.0 / 3000000.0)
        step = int(np.sign(x)) * int(np.floor(abs(x) + 0.5))
        assert gps.carrier_advance_u32(7, f, 3) == float((7 + 3 * step) % TWO32)


@pytest.mark.parametrize("ranks", [2, 4, 8])
def test_link_apply_nco_composes_to_the_sequential_closed_form(ranks, tmp_path):
    """U32 links are exact: composing the links of K slices gives, for every cut, the sequential u32 chain."""
    ch, _ = gps.scenario(make_nav(tmp_path, 32), *LOC60, seconds=310, max_chan=32, start=START, carrier="u32")
    edges = event_edges(ch, ranks)
    nchan = ch.shape[1]
    # sequential closed form, block by block
    seq = {}
    u, prev = np.zeros(nchan), np.zeros(nchan, np.int32)
    for b in range(ch.shape[0]):
        row = ch[b]
        for c in range(nchan):
            if row["prn"][c] <= 0:
                u[c] = 0.0
                continue
            start = u[c] if row["prn"][c] == prev[c] else row["carr_phase"][c]
            u[c] = gps.carrier_advance_u32(start, row["f_carr"][c], gps.BLOCK_SAMPLES)
        prev = np.where(row["prn"] > 0, row["prn"], 0)
        seq[b + 1] = (prev.copy(), u.copy())
    prn, ph = None, None
    for lo, hi in zip(edges[:-1], edges[1:]):
        link = gps.slice_link_host(ch[lo:hi], carrier="u32")
        prn, ph = gps.link_apply(link, nchan, prn, ph, carrier="u32")
        assert np.array_equal(prn, seq[hi][0]), hi
        assert np.array_equal(ph, seq[hi][1]), hi
    with pytest.raises(gps.GpsB200Error):
        gps.link_apply(link, nchan, prn, ph + 0.5, carrier="u32")


# ======================================================================================================================
# GPU
# ======================================================================================================================
def synth(ch, nav, ss, max_blocks=None, **kw):
    with gps.Context(ch.shape[1], max_blocks or ch.shape[0], max_nav_frames=len(nav), carrier="u32", **kw) as ctx:
        ctx.set_nav_frames(nav)
        out, cp, st = ctx.synth_blocks(ch, ss, want_stats=True)
        return out, cp, st, ctx.synth_kernel_name(ch.shape[1])


def want_crcs(g):
    c = g["crcs"]
    return c if c.ndim == 1 else c[:, 0]          # CRC-only fixtures hold the whole-block CRCs alone


def assert_crcs(out, g, what):
    crc = scenario.crc_blocks(out)
    bad = np.nonzero(crc != want_crcs(g)[:crc.size])[0]
    assert bad.size == 0, "%s: %d/%d blocks differ, first %s" % (what, bad.size, crc.size, bad[:5])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sky12_static_10s_i8_u32", "sky32_static_10s_i8_u32", "sky12_circle_60s_i16_u32"])
def test_u32_golden_streams_from_dumped_parameters(name):
    g = scenario.load_golden(name)
    ch, frames = scenario.golden_chans(g)
    out, cp, st, kname = synth(ch, frames, int(g["sample_size"]))
    assert kname == "k_synth_lanes_u32"
    assert_crcs(out, g, name)
    for i, blk in zip(g["keep_idx"], g["keep_blocks"]):
        assert np.array_equal(out[i * gps.BLOCK_ELEMS:(i + 1) * gps.BLOCK_ELEMS], blk)


@pytest.mark.gpu
@pytest.mark.parametrize("name,nsat,secs,loc,motion", [("sky12_static_10s_i8_u32", 12, 10, LOC, None),
                                                       ("sky12_circle_60s_i16_u32", 12, 60, LOC, CIRCLE),
                                                       ("sky32_lat60_310s_i8_u32", 32, 310, LOC60, None),
                                                       ("sky32_static_600s_i8_u32", 32, 600, LOC, None)])
def test_u32_golden_streams_from_the_rinex_file(name, nsat, secs, loc, motion, tmp_path):
    g = scenario.load_golden(name)
    ch, nav = gps.scenario(make_nav(tmp_path, nsat), *loc, seconds=secs, max_chan=nsat, start=START,
                           motion_file=motion, carrier="u32")
    assert ch.shape[0] == g["crcs"].shape[0]
    if ch.shape[0] <= 3000:
        assert_crcs(synth(ch, nav, int(g["sample_size"]))[0], g, name)
    else:                        # longer than one context call: consecutive calls chained by carr_phase_out
        outs, cp = [], None
        with gps.Context(nsat, 3000, max_nav_frames=len(nav), carrier="u32") as ctx:
            ctx.set_nav_frames(nav)
            for b0 in range(0, ch.shape[0], 3000):
                part = ch[b0:b0 + 3000].copy()
                if cp is not None:
                    cont = (part["prn"][0] > 0) & (part["prn"][0] == ch["prn"][b0 - 1])
                    part["carr_phase"][0][cont] = cp[cont]
                o, cp = ctx.synth_blocks(part, 1)
                outs.append(scenario.crc_blocks(o))
        crc = np.concatenate(outs)
        bad = np.nonzero(crc != want_crcs(g))[0]
        assert bad.size == 0, bad[:10]


@pytest.mark.gpu
@pytest.mark.parametrize("iq16", [False, True])
def test_u32_cli_writes_the_integer_reference_stream(iq16, tmp_path):
    """gpsb200-sim --u32-carrier, int8 (configs[1]) and int16 (the circle.csv motion run); --gpus 2 where two devices
    exist."""
    import torch
    exe = os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "gpsb200-sim")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(scenario.ROOT, "multi-sdr-gps-sim_b200", "csrc")])
    name = "sky12_circle_60s_i16_u32" if iq16 else "sky12_static_10s_i8_u32"
    g = scenario.load_golden(name)
    cmd = [exe, "-e", make_nav(tmp_path, 12), "-l", "%r,%r,%r" % LOC, "-s", "2024/01/07,02:00:00", "--u32-carrier"]
    cmd += ["--iq16", "-m", CIRCLE, "-d", "60"] if iq16 else ["-d", "10"]
    for n in [1] + ([2] if torch.cuda.device_count() >= 2 else []):
        out = tmp_path / ("iq_%d.bin" % n)
        subprocess.check_call(cmd + ["--gpus", str(n), "-o", str(out)])
        s = np.fromfile(out, dtype=np.int16 if iq16 else np.int8)
        assert s.size == g["crcs"].shape[0] * gps.BLOCK_ELEMS
        assert_crcs(s, g, "cli --gpus %d" % n)


@pytest.mark.gpu
@pytest.mark.parametrize("nchan,ss", [(1, 1), (5, 2), (12, 1), (16, 2), (17, 1), (32, 1), (32, 2)])
def test_u32_synthetic_vs_oracle_both_kernels(nchan, ss, monkeypatch):
    """Seeded synthetic parameters against oracle_synth_block_u32 with k_synth_lanes_u32, with k_synth_u32
    (GPSB200_LANES=0), and with a run length the lanes kernel does not take (fallback to k_synth_u32)."""
    ch, nav = u32_synthetic(5, nchan, seed=300 + nchan)
    ch["carr_phase"][0, 0] = TWO32 - 7
    want, carr = oracle_run_u32(ch, nav, ss)
    for lanes_on, run, name in (("1", 0, "k_synth_lanes_u32"), ("0", 0, "k_synth_u32"), ("1", 800, "k_synth_u32")):
        monkeypatch.setenv("GPSB200_LANES", lanes_on)
        out, cp, st, kname = synth(ch, nav, ss, run_samples=run)
        assert kname == name
        assert np.array_equal(out, want), name
        assert np.array_equal(cp, carr), name


@pytest.mark.gpu
def test_u32_call_paths_equal_one_call():
    """Split calls, one-block calls (the drop-in cadence), the device path and the scatter path equal one whole call;
    a U32 call launches no probe kernel, walks nothing on the host, and launches fewer kernels than an FP64 call."""
    import torch
    g = scenario.load_golden("sky12_static_10s_i8_u32")
    ch, nav = scenario.golden_chans(g)
    nblk, nchan = ch.shape
    whole, cp_whole, st_u, _ = synth(ch, nav, 1)
    assert_crcs(whole, g, "whole")
    assert st_u.probe_kernel_ms == 0.0 and st_u.chain_fallbacks == 0
    with gps.Context(nchan, nblk, max_nav_frames=len(nav)) as ctx:          # same blocks, FP64 mode
        ctx.set_nav_frames(nav)
        f64 = ch.copy()
        f64["carr_phase"] = (ch["carr_phase"] / TWO32)
        _, _, st_f = ctx.synth_blocks(f64, 1, want_stats=True)
    assert st_u.launches < st_f.launches, (st_u.launches, st_f.launches)
    with gps.Context(nchan, nblk, max_nav_frames=len(nav), carrier="u32") as ctx:
        ctx.set_nav_frames(nav)
        for cuts in ([0, 40, 99], [0, 1, 2, 3, 50, 97, 99], list(range(nblk + 1))):      # last: one block per call
            outs, cp = [], None
            for lo, hi in zip(cuts[:-1], cuts[1:]):
                part = ch[lo:hi].copy()
                if cp is not None:
                    part["carr_phase"][0] = np.where(part["prn"][0] == ch["prn"][lo - 1], cp, part["carr_phase"][0])
                o, cp = ctx.synth_blocks(part, 1)
                outs.append(o)
            assert np.array_equal(np.concatenate(outs), whole), cuts
            assert np.array_equal(cp, cp_whole)
        dev = torch.empty(nblk * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
        cp_dev, st_d = ctx.synth_blocks_device(ch, 1, dev.data_ptr(), want_stats=True)
        torch.cuda.synchronize()
        assert np.array_equal(dev.cpu().numpy(), whole) and np.array_equal(cp_dev, cp_whole)
        assert st_d.probe_kernel_ms == 0.0 and st_d.chain_fallbacks == 0
        bufs = [np.empty(gps.BLOCK_ELEMS, np.int8) for _ in range(nblk)]
        ptrs = (C.c_void_p * nblk)(*[b.ctypes.data for b in bufs])
        cps = np.zeros(nchan)
        rc = gps.lib().gpsb200_synth_blocks_scatter(ctx._h, ch.ctypes.data, nblk, nchan, 1, ptrs, cps.ctypes.data, None)
        assert rc == 0
        assert np.array_equal(np.concatenate(bufs), whole) and np.array_equal(cps, cp_whole)
        with pytest.raises(gps.GpsB200Error):
            ctx.debug_corrupt_chain(True)                # no carrier chain to corrupt
        bad = ch.copy()
        bad["carr_phase"][0, 3] = 0.25                   # not a u32 phase
        with pytest.raises(gps.GpsB200Error):
            ctx.synth_blocks(bad, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [2, 4, 8])
@pytest.mark.parametrize("dst_host", [False, True])
def test_u32_three_step_slices_equal_the_integer_reference_stream(ranks, dst_host, tmp_path):
    """gpsb200_slice_prepare / _probe / _finish over K "ranks" of the 310 s reallocation scenario, cut also exactly where
    a satellite rises or sets: the links compose to the EXACT incoming states (no speculation), the concatenation is
    the integer reference's stream, and the final state is the one-call state."""
    import torch
    g = scenario.load_golden("sky32_lat60_310s_i8_u32")
    ch, nav = gps.scenario(make_nav(tmp_path, 32), *LOC60, seconds=310, max_chan=32, start=START, carrier="u32")
    edges = event_edges(ch, ranks)
    nchan = ch.shape[1]
    ctxs, outs, links = [], [], []
    try:
        for lo, hi in zip(edges[:-1], edges[1:]):
            ctx = gps.Context(nchan, hi - lo, max_nav_frames=len(nav), carrier="u32")
            ctx.set_nav_frames(nav)
            ctxs.append(ctx)
            if dst_host:
                o = torch.empty((hi - lo) * gps.BLOCK_ELEMS, dtype=torch.int8).pin_memory().numpy()
                outs.append(o)
                links.append(ctx.slice_prepare(ch[lo:hi], 1, dst_host=o))
            else:
                o = torch.empty((hi - lo) * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
                outs.append(o)
                links.append(ctx.slice_prepare(ch[lo:hi], 1, o.data_ptr()))
        prn, ph, guesses = None, None, []
        for k, (ctx, link) in enumerate(zip(ctxs, links)):
            ctx.slice_probe(prn, ph, eager=k + 1 < len(ctxs))
            guesses.append((prn, ph))
            prn, ph = gps.link_apply(link, nchan, prn, ph, carrier="u32")
        prn, ph = None, None
        for k, ctx in enumerate(ctxs):
            if k > 0:          # the composed links were exact
                assert np.array_equal(guesses[k][0], prn) and np.array_equal(guesses[k][1], ph), k
            handed = []
            prn, ph, st = ctx.slice_finish(prn, ph, want_stats=True, handoff=lambda a, b: handed.append((a, b)))
            assert len(handed) == 1 and np.array_equal(handed[0][1], ph)
            assert st.chain_fallbacks == 0
        for ctx in ctxs:
            ctx.slice_wait()
        torch.cuda.synchronize()
        crc = np.concatenate([scenario.crc_blocks(o if dst_host else o.cpu().numpy()) for o in outs])
        bad = np.nonzero(crc != want_crcs(g))[0]
        assert bad.size == 0, (edges, bad[:10])
    finally:
        for ctx in ctxs:
            ctx.close()
    with gps.Context(nchan, ch.shape[0], max_nav_frames=len(nav), carrier="u32") as ctx:
        assert np.array_equal(ctx.carrier_chain(ch), ph)


@pytest.mark.gpu
@pytest.mark.ref
def test_reference_program_with_the_drop_in_patch_on_the_integer_build(tmp_path):
    """oracle/_ref/ref_gpsb200_12_u32: the reference program built without FLOAT_CARR_PHASE, sample loop replaced by
    gpsb200_synth_blocks in a GPSB200_CARRIER_U32 context (integration_setup_u32.inc): configs[1], all 99 blocks equal
    the integer reference's enqueue stream."""
    exe = os.path.join(scenario.ROOT, "oracle", "_ref", "ref_gpsb200_12_u32")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/ref_gpsb200_12_u32 not built (needs the reference sources)")
    g = scenario.load_golden("sky12_static_10s_i8_u32")
    r = subprocess.run([exe, "-e", make_nav(tmp_path, 12), "-l", "%r,%r,%r" % LOC, "-d", "10"], cwd=tmp_path,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-600:]
    s = np.fromfile(tmp_path / "iqdata.bin", dtype=np.int8)
    assert s.size == 99 * gps.BLOCK_ELEMS, s.size
    assert_crcs(s, g, "ref_gpsb200_12_u32")
