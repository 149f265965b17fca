"""The reference program exactly as shipped (own fifo.c / sdr_iqfile.c) against the golden
enqueue stream: its iqdata.bin is the stream with blocks 1..6 missing (fifo.c:163-168).
The block digests of that iqdata.bin are stored in tests/golden (make_golden.py runs the
stock program oracle/_ref/ref_stock12 where the reference sources are available)."""
import os
import subprocess

import numpy as np
import pytest

import scenario


def test_stock_iqfile_is_enqueue_stream_minus_blocks_1_to_6():
    s = scenario.load_golden("sky12_static_10s_stock_iqfile")["crcs"]
    g = scenario.load_golden("sky12_static_10s_i8")
    keep = [0] + list(range(7, 99))
    assert s.size == len(keep)
    for crc, b in zip(s, keep):
        assert crc == g["crcs"][b, 0], b


@pytest.mark.ref
@pytest.mark.parametrize("bits", [8, 16])
def test_reference_sink_code_runs_unmodified_on_our_fifo(bits, tmp_path):
    """Drop-in claim of INTEGRATION.md section 3, compiled and run: the reference's own sdr.c (dispatch table,
    sdr.c:35-87) and sdr_iqfile.c (writer thread, sdr_iqfile.c:22-77) are built unmodified and linked with
    libgpsb200.so INSTEAD OF fifo.o (oracle/Makefile: ref_sinkfeed). A producer replays a stream through
    fifo_acquire / fifo_enqueue exactly as gps_thread_ep does; the sink's iqdata.bin must be that stream --
    all of it (the stock fifo.c would lose buffers 1..6, fifo.c:163-168)."""
    exe = os.path.join(scenario.ROOT, "oracle", "_ref", "ref_sinkfeed")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(scenario.ROOT, "oracle")])
    rng = np.random.default_rng(bits)
    dt = np.int8 if bits == 8 else np.int16
    info = np.iinfo(dt)
    stream = rng.integers(info.min, info.max + 1, size=23 * 600000, dtype=dt)
    src = tmp_path / "in.bin"
    stream.tofile(src)
    out = subprocess.run([exe, str(src), str(bits)], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-400:]
    got = np.fromfile(tmp_path / "iqdata.bin", dtype=dt)
    assert got.size == stream.size and np.array_equal(got, stream)
