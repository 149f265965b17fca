"""ctypes mirror of include/gpsb200.h. No compute happens here and there is no CPU
fallback: if libgpsb200.so is missing or no CUDA device is present the calls fail."""
import ctypes as C
import math
import os

import numpy as np

BLOCK_SAMPLES = 300000
BLOCK_ELEMS = 600000
SC08, SC16 = 1, 2
CARRIER_FP64, CARRIER_U32 = 0, 1     # gpsb200_config_t.carrier_nco
_CARRIER = {"fp64": CARRIER_FP64, "u32": CARRIER_U32}


def carrier_nco(carrier):
    """'fp64' | 'u32' (or the GPSB200_CARRIER_* value) -> GPSB200_CARRIER_* value."""
    if isinstance(carrier, str):
        if carrier not in _CARRIER:
            raise ValueError("carrier must be 'fp64' or 'u32', not %r" % carrier)
        return _CARRIER[carrier]
    if carrier not in (CARRIER_FP64, CARRIER_U32):
        raise ValueError("bad carrier NCO %r" % (carrier,))
    return int(carrier)

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path():
    return os.path.join(_HERE, "libgpsb200.so")


class GpsB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("gpsb200 error %d: %s" % (code, msg))
        self.code = code


class Chan(C.Structure):
    """gpsb200_chan_t (64 bytes)."""
    _fields_ = [("prn", C.c_int32), ("iword", C.c_int32), ("ibit", C.c_int32), ("icode", C.c_int32),
                ("nav_frame", C.c_int32), ("reserved", C.c_int32),
                ("f_carr", C.c_double), ("f_code", C.c_double), ("carr_phase", C.c_double),
                ("code_phase", C.c_double), ("gain", C.c_double)]


CHAN_DTYPE = np.dtype([("prn", "<i4"), ("iword", "<i4"), ("ibit", "<i4"), ("icode", "<i4"),
                       ("nav_frame", "<i4"), ("reserved", "<i4"),
                       ("f_carr", "<f8"), ("f_code", "<f8"), ("carr_phase", "<f8"),
                       ("code_phase", "<f8"), ("gain", "<f8")])
assert CHAN_DTYPE.itemsize == C.sizeof(Chan) == 64


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_chan", C.c_int32), ("max_blocks", C.c_int32),
                ("max_nav_frames", C.c_int32), ("host_threads", C.c_int32), ("run_samples", C.c_int32),
                ("carrier_nco", C.c_int32)]


class ScenarioConfig(C.Structure):
    _fields_ = [("nav_file", C.c_char_p), ("motion_file", C.c_char_p),
                ("lat_deg", C.c_double), ("lon_deg", C.c_double), ("height_m", C.c_double),
                ("duration_ds", C.c_int32), ("max_chan", C.c_int32), ("ionosphere_enable", C.c_int32),
                ("pluto_gain", C.c_int32),
                ("start_year", C.c_int32), ("start_month", C.c_int32), ("start_day", C.c_int32),
                ("start_hour", C.c_int32), ("start_min", C.c_int32), ("rinex3", C.c_int32),
                ("start_sec", C.c_double), ("target_valid", C.c_int32), ("carrier_u32", C.c_int32),
                ("target_distance_m", C.c_double), ("target_bearing_deg", C.c_double), ("target_height_m", C.c_double),
                ("almanac_file", C.c_char_p)]


class SliceLink(C.Structure):
    """gpsb200_slice_link_t."""
    _fields_ = [("prn_first", C.c_int32 * 32), ("prn_last", C.c_int32 * 32), ("reset_inside", C.c_int32 * 32),
                ("first_phase", C.c_double * 32), ("value", C.c_double * 32)]


class Stats(C.Structure):
    _fields_ = [("host_chain_ms", C.c_double), ("h2d_ms", C.c_double), ("kernel_ms", C.c_double),
                ("d2h_ms", C.c_double), ("checkpoint_kernel_ms", C.c_double), ("synth_kernel_ms", C.c_double),
                ("probe_kernel_ms", C.c_double),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("launches", C.c_int32),
                ("chain_fallbacks", C.c_int32)]


HANDOFF_FN = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_double))     # gpsb200_handoff_fn

_lib = None

EXPORTS = ["gpsb200_create", "gpsb200_destroy", "gpsb200_last_error", "gpsb200_version", "gpsb200_set_nav",
           "gpsb200_synth_blocks", "gpsb200_synth_blocks_scatter", "gpsb200_synth_blocks_device", "gpsb200_replay_device",
           "gpsb200_carrier_advance", "gpsb200_carrier_chain", "gpsb200_carrier_chain_device", "gpsb200_carrier_probe_fixup",
           "gpsb200_codegen", "gpsb200_bind_numa", "gpsb200_span_chain_host", "gpsb200_lanes_model_block", "gpsb200_slice_prepare", "gpsb200_slice_probe",
           "gpsb200_slice_finish", "gpsb200_slice_finish_cb", "gpsb200_slice_wait", "gpsb200_link_apply", "gpsb200_slice_link_host",
           "gpsb200_link_apply_nco", "gpsb200_slice_link_host_nco", "gpsb200_debug_corrupt_chain", "gpsb200_synth_kernel_name",
           "gpsb200_scenario_create", "gpsb200_scenario_destroy", "gpsb200_scenario_error",
           "gpsb200_scenario_blocks", "gpsb200_scenario_channels", "gpsb200_scenario_nav_frames",
           "gpsb200_scenario_chans", "gpsb200_scenario_nav",
           "fifo_create", "fifo_destroy", "fifo_wait_next", "fifo_wait_full", "fifo_halt", "fifo_acquire",
           "fifo_enqueue", "fifo_dequeue", "fifo_release", "fifo_set_compat_drop",
           "gpsb200_iqfile_start", "gpsb200_iqfile_stop", "gpsb200_fifo_push", "gpsb200_fifo_push_flush"]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(lib_path()):
            raise GpsB200Error(-2, "libgpsb200.so not built (run __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(lib_path())
        L.gpsb200_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.gpsb200_destroy.argtypes = [C.c_void_p]
        L.gpsb200_last_error.argtypes = [C.c_void_p]
        L.gpsb200_last_error.restype = C.c_char_p
        L.gpsb200_version.restype = C.c_char_p
        L.gpsb200_set_nav.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.gpsb200_synth_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.POINTER(Stats)]
        L.gpsb200_synth_blocks_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.POINTER(Stats)]
        L.gpsb200_replay_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gpsb200_carrier_advance.argtypes = [C.c_double, C.c_double, C.c_int64]
        L.gpsb200_carrier_advance.restype = C.c_double
        L.gpsb200_codegen.argtypes = [C.c_int, C.c_void_p]
        L.gpsb200_scenario_create.argtypes = [C.POINTER(ScenarioConfig), C.POINTER(C.c_void_p)]
        L.gpsb200_scenario_destroy.argtypes = [C.c_void_p]
        L.gpsb200_scenario_error.argtypes = [C.c_void_p]
        L.gpsb200_scenario_error.restype = C.c_char_p
        for fn in ("blocks", "channels", "nav_frames"):
            getattr(L, "gpsb200_scenario_" + fn).argtypes = [C.c_void_p]
        L.gpsb200_scenario_chans.argtypes = [C.c_void_p]
        L.gpsb200_scenario_chans.restype = C.c_void_p
        L.gpsb200_scenario_nav.argtypes = [C.c_void_p]
        L.gpsb200_scenario_nav.restype = C.c_void_p
        L.gpsb200_carrier_probe_fixup.argtypes = [C.c_double, C.c_double, C.c_double, C.c_int64, C.POINTER(C.c_double)]
        L.gpsb200_carrier_chain_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.gpsb200_carrier_chain.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.gpsb200_span_chain_host.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.gpsb200_slice_prepare.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.POINTER(SliceLink)]
        L.gpsb200_slice_finish_cb.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Stats),
                                              HANDOFF_FN, C.c_void_p]
        L.gpsb200_slice_wait.argtypes = [C.c_void_p]
        L.gpsb200_slice_link_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(SliceLink)]
        L.gpsb200_slice_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.gpsb200_slice_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Stats)]
        L.gpsb200_link_apply.argtypes = [C.POINTER(SliceLink), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gpsb200_slice_link_host_nco.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(SliceLink)]
        L.gpsb200_link_apply_nco.argtypes = [C.POINTER(SliceLink), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p]
        L.gpsb200_debug_corrupt_chain.argtypes = [C.c_void_p, C.c_int]
        L.gpsb200_synth_kernel_name.argtypes = [C.c_void_p, C.c_int]
        L.gpsb200_synth_kernel_name.restype = C.c_char_p
        _lib = L
    return _lib


def bind_numa(device=0):
    """gpsb200_bind_numa: pin the calling thread (and threads created later) to the GPU's NUMA node. -> node or -1."""
    L = lib()
    L.gpsb200_bind_numa.argtypes = [C.c_int]
    L.gpsb200_bind_numa.restype = C.c_int
    return int(L.gpsb200_bind_numa(int(device)))


def codegen(prn):
    ca = np.zeros(1023, np.uint8)
    rc = lib().gpsb200_codegen(prn, ca.ctypes.data)
    if rc:
        raise GpsB200Error(rc, "gpsb200_codegen(%d)" % prn)
    return ca


def carrier_advance(phase, f_carr, nsamples):
    return lib().gpsb200_carrier_advance(float(phase), float(f_carr), int(nsamples))


def carrier_chain(chans, phase_in=None, threads=16):
    """Exact carrier phase of every slot after all blocks of chans[nblk, nchan] (host only)."""
    a = np.ascontiguousarray(chans, dtype=CHAN_DTYPE)
    nblk, nchan = a.shape
    out = np.zeros(nchan, np.float64)
    pin = None if phase_in is None else np.ascontiguousarray(phase_in, dtype=np.float64)
    rc = lib().gpsb200_carrier_chain(a.ctypes.data, nblk, nchan, None if pin is None else pin.ctypes.data,
                                     out.ctypes.data, threads)
    if rc:
        raise GpsB200Error(rc, "gpsb200_carrier_chain")
    return out


def lanes_model_block(chans_row, nav_frame, run_samples=2400, force=0, carrier="fp64"):
    """Host model of the lane = sample kernel for one block. chans_row: CHAN_DTYPE[nchan]; nav_frame: uint32[nchan, 60].
    carrier='u32' sets force bit 16 (integer carrier NCO). -> (iq int16[600000], carr_out float64[nchan], counters int64[4])"""
    if carrier_nco(carrier) == CARRIER_U32:
        force |= 16
    a = np.ascontiguousarray(chans_row, dtype=CHAN_DTYPE)
    nv = np.ascontiguousarray(nav_frame, dtype=np.uint32)
    iq = np.zeros(BLOCK_ELEMS, np.int16)
    co = np.zeros(a.size, np.float64)
    cnt = np.zeros(4, np.int64)
    L = lib()
    L.gpsb200_lanes_model_block.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    rc = L.gpsb200_lanes_model_block(a.ctypes.data, a.size, nv.ctypes.data, run_samples, force, iq.ctypes.data, co.ctypes.data,
                                     cnt.ctypes.data)
    if rc:
        raise GpsB200Error(rc, "gpsb200_lanes_model_block")
    return iq, co, cnt


def span_chain_host(f_carr, start_true, start_guess):
    """Host model of the two-level chain for one span. -> float64[nblk + 1] exact block starts + end, or None if
    the span-level speculation was rejected."""
    f = np.ascontiguousarray(f_carr, dtype=np.float64)
    out = np.zeros(f.size + 1)
    rc = lib().gpsb200_span_chain_host(f.ctypes.data, f.size, float(start_true), float(start_guess), out.ctypes.data)
    if rc < 0:
        raise GpsB200Error(rc, "gpsb200_span_chain_host")
    return out if rc == 1 else None


def slice_link_host(chans, carrier="fp64"):
    """gpsb200_slice_link_host_nco: the closed-form link of a slice (host only; exact for carrier='u32'). -> SliceLink"""
    a = np.ascontiguousarray(chans, dtype=CHAN_DTYPE)
    link = SliceLink()
    rc = lib().gpsb200_slice_link_host_nco(a.ctypes.data, a.shape[0], a.shape[1], carrier_nco(carrier), C.byref(link))
    if rc:
        raise GpsB200Error(rc, "gpsb200_slice_link_host_nco")
    return link


def link_apply(link, nchan, prn_in=None, phase_in=None, carrier="fp64"):
    """gpsb200_link_apply_nco -> (prn_out int32[nchan], phase_out float64[nchan])."""
    pi = None if prn_in is None else np.ascontiguousarray(prn_in, dtype=np.int32)
    xi = None if phase_in is None else np.ascontiguousarray(phase_in, dtype=np.float64)
    po, xo = np.zeros(nchan, np.int32), np.zeros(nchan, np.float64)
    rc = lib().gpsb200_link_apply_nco(C.byref(link), nchan, carrier_nco(carrier), None if pi is None else pi.ctypes.data,
                                      None if xi is None else xi.ctypes.data, po.ctypes.data, xo.ctypes.data)
    if rc:
        raise GpsB200Error(rc, "gpsb200_link_apply_nco")
    return po, xo


def carrier_advance_u32(u, f_carr, n):
    """The reference's integer carrier NCO (gps.c:2746, 2828) on the host, for tests: u + n * carr_phasestep modulo
    2^32, carr_phasestep = (int) round(512.0 * 65536.0 * f_carr * delt) evaluated in the reference's order."""
    return float((int(u) + int(n) * _u32_step(f_carr)) % (1 << 32))


def _u32_step(f_carr):
    x = (33554432.0 * float(f_carr)) * (1.0 / 3000000.0)
    ax = abs(x)
    r = math.floor(ax)
    r += 1 if ax - r >= 0.5 else 0                       # C round(): ties away from zero (ax - r is exact)
    return int(r) if x >= 0 else -int(r)


def scenario(nav_file, lat, lon, height, seconds, max_chan=12, motion_file=None, start=None,
             ionosphere=True, pluto_gain=False, rinex3=False, target=None, carrier="fp64", almanac=None):
    """Run the host scenario engine. -> (chans[nblk, max_chan] CHAN_DTYPE, nav[nframes, max_chan, 60] uint32).
    start: (y, m, d, hh, mm, sec) or None for the first ephemeris epoch. carrier='u32': allocation phases of the
    reference's integer carrier build (u32 accumulators). almanac: path of a SEM almanac file whose records fill the
    almanac pages of subframes 4 and 5, as the reference does with its almanac.sem; None: no almanac pages."""
    cfg = ScenarioConfig()
    cfg.nav_file = os.fsencode(nav_file)
    cfg.motion_file = os.fsencode(motion_file) if motion_file else None
    cfg.lat_deg, cfg.lon_deg, cfg.height_m = lat, lon, height
    cfg.duration_ds = int(seconds * 10.0 + 0.5)
    cfg.max_chan = max_chan
    cfg.ionosphere_enable = 1 if ionosphere else 0
    cfg.pluto_gain = 1 if pluto_gain else 0
    cfg.rinex3 = 1 if rinex3 else 0
    cfg.carrier_u32 = 1 if carrier_nco(carrier) == CARRIER_U32 else 0
    cfg.almanac_file = os.fsencode(almanac) if almanac is not None else None
    if target is not None:          # -t distance,bearing,height
        cfg.target_valid = 1
        cfg.target_distance_m, cfg.target_bearing_deg, cfg.target_height_m = [float(v) for v in target]
    if start:
        (cfg.start_year, cfg.start_month, cfg.start_day, cfg.start_hour, cfg.start_min) = [int(v) for v in start[:5]]
        cfg.start_sec = float(start[5])
    h = C.c_void_p()
    L = lib()
    rc = L.gpsb200_scenario_create(C.byref(cfg), C.byref(h))
    try:
        if rc:
            raise GpsB200Error(rc, L.gpsb200_scenario_error(h).decode() if h else "gpsb200_scenario_create")
        nblk, nch, nfr = (L.gpsb200_scenario_blocks(h), L.gpsb200_scenario_channels(h),
                          L.gpsb200_scenario_nav_frames(h))
        chans = np.frombuffer(C.string_at(L.gpsb200_scenario_chans(h), nblk * nch * 64), dtype=CHAN_DTYPE)
        nav = np.frombuffer(C.string_at(L.gpsb200_scenario_nav(h), nfr * nch * 60 * 4), dtype=np.uint32)
        return chans.reshape(nblk, nch).copy(), nav.reshape(nfr, nch, 60).copy()
    finally:
        if h:
            L.gpsb200_scenario_destroy(h)


class Context:
    """gpsb200_ctx_t. `chans` arguments are numpy arrays of CHAN_DTYPE shaped [nblk, nchan]."""

    def __init__(self, max_chan, max_blocks, device=0, max_nav_frames=1, host_threads=0, run_samples=0, carrier="fp64"):
        """carrier: 'fp64' (the reference as shipped) or 'u32' (its integer carrier NCO build); in a 'u32' context
        every carrier phase in or out is the u32 accumulator as an integer-valued float."""
        self._h = C.c_void_p()
        self.carrier = "u32" if carrier_nco(carrier) == CARRIER_U32 else "fp64"
        self.cfg = Config(device, max_chan, max_blocks, max_nav_frames, host_threads, run_samples, carrier_nco(carrier))
        rc = lib().gpsb200_create(C.byref(self.cfg), C.byref(self._h))
        if rc:
            msg = lib().gpsb200_last_error(self._h).decode() if self._h else "gpsb200_create: bad configuration"
            if self._h:
                lib().gpsb200_destroy(self._h)
                self._h = C.c_void_p()
            raise GpsB200Error(rc, msg)

    def close(self):
        if self._h:
            lib().gpsb200_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc:
            raise GpsB200Error(rc, lib().gpsb200_last_error(self._h).decode())

    def set_nav(self, frame, chan, words):
        w = np.ascontiguousarray(words, dtype=np.uint32)
        assert w.size == 60
        self._check(lib().gpsb200_set_nav(self._h, frame, chan, w.ctypes.data))

    def set_nav_frames(self, frames):
        """frames: uint32[nframes, nchan, 60]."""
        for f in range(frames.shape[0]):
            for c in range(frames.shape[1]):
                self.set_nav(f, c, frames[f, c])

    @staticmethod
    def _chans(chans):
        a = np.ascontiguousarray(chans, dtype=CHAN_DTYPE)
        assert a.ndim == 2
        return a

    def synth_blocks(self, chans, sample_size=SC08, out=None, want_stats=False):
        """Host-destination path (H2D params + kernels + D2H result). Returns (iq, carr_phase_out[, Stats])."""
        a = self._chans(chans)
        nblk, nchan = a.shape
        dt = np.int16 if sample_size == SC16 else np.int8
        if out is None:
            out = np.empty(nblk * BLOCK_ELEMS, dt)
        assert out.dtype == dt and out.size >= nblk * BLOCK_ELEMS and out.flags.c_contiguous
        cp = np.zeros(nchan, np.float64)
        st = Stats()
        self._check(lib().gpsb200_synth_blocks(self._h, a.ctypes.data, nblk, nchan, sample_size,
                                               out.ctypes.data, cp.ctypes.data, C.byref(st)))
        return (out, cp, st) if want_stats else (out, cp)

    def synth_blocks_device(self, chans, sample_size, dst_ptr, stream=0, want_stats=False):
        """Device-destination path: dst_ptr is a raw device pointer (e.g. torch tensor .data_ptr())."""
        a = self._chans(chans)
        nblk, nchan = a.shape
        cp = np.zeros(nchan, np.float64)
        st = Stats()
        self._check(lib().gpsb200_synth_blocks_device(self._h, a.ctypes.data, nblk, nchan, sample_size,
                                                      C.c_void_p(dst_ptr), C.c_void_p(stream), cp.ctypes.data,
                                                      C.byref(st) if want_stats else None))
        return (cp, st) if want_stats else cp

    def slice_prepare(self, chans, sample_size, dst_ptr=0, stream=0, dst_host=None):
        """Step 1 of the time-slice hand-over. dst_ptr: raw device pointer and/or dst_host: numpy array in pinned
        memory. -> SliceLink"""
        a = self._chans(chans)
        nblk, nchan = a.shape
        link = SliceLink()
        hp = None if dst_host is None else C.c_void_p(dst_host.ctypes.data)
        self._check(lib().gpsb200_slice_prepare(self._h, a.ctypes.data, nblk, nchan, sample_size, C.c_void_p(dst_ptr),
                                                hp, C.c_void_p(stream), C.byref(link)))
        self._slice_nchan = nchan
        return link

    def slice_probe(self, prn_in=None, phase_guess_in=None, eager=False):
        """Step 2. eager: all speculative work up front (a successor is waiting for this slice's outgoing state)."""
        pi = None if prn_in is None else np.ascontiguousarray(prn_in, dtype=np.int32)
        xi = None if phase_guess_in is None else np.ascontiguousarray(phase_guess_in, dtype=np.float64)
        self._check(lib().gpsb200_slice_probe(self._h, None if pi is None else pi.ctypes.data,
                                              None if xi is None else xi.ctypes.data, 1 if eager else 0))

    def slice_finish(self, prn_in=None, phase_in=None, want_stats=False, handoff=None):
        """Step 3. -> (prn_out, phase_out[, Stats]): the exact chain state after the slice. handoff(prn, phase), if
        given, is called with that state as soon as the host scan has it -- for an eager slice before the long kernels
        are enqueued (gpsb200_slice_finish_cb)."""
        n = self._slice_nchan
        pi = None if prn_in is None else np.ascontiguousarray(prn_in, dtype=np.int32)
        xi = None if phase_in is None else np.ascontiguousarray(phase_in, dtype=np.float64)
        po, xo = np.zeros(n, np.int32), np.zeros(n, np.float64)
        st = Stats()

        def _cb(_user, p_prn, p_ph):
            handoff(np.ctypeslib.as_array(p_prn, shape=(n,)).copy(), np.ctypeslib.as_array(p_ph, shape=(n,)).copy())

        cb = HANDOFF_FN(_cb) if handoff is not None else C.cast(None, HANDOFF_FN)
        self._check(lib().gpsb200_slice_finish_cb(self._h, None if pi is None else pi.ctypes.data,
                                                  None if xi is None else xi.ctypes.data, po.ctypes.data, xo.ctypes.data,
                                                  C.byref(st), cb, None))
        return (po, xo, st) if want_stats else (po, xo)

    def slice_wait(self):
        self._check(lib().gpsb200_slice_wait(self._h))

    def synth_kernel_name(self, nchan):
        return lib().gpsb200_synth_kernel_name(self._h, int(nchan)).decode()

    def debug_corrupt_chain(self, on):
        self._check(lib().gpsb200_debug_corrupt_chain(self._h, 1 if on else 0))

    def carrier_chain(self, chans, phase_in=None):
        """Exact carrier phases after all blocks of chans (device probe + host fix-up, no synthesis)."""
        a = self._chans(chans)
        nblk, nchan = a.shape
        out = np.zeros(nchan, np.float64)
        pin = None if phase_in is None else np.ascontiguousarray(phase_in, dtype=np.float64)
        self._check(lib().gpsb200_carrier_chain_device(self._h, a.ctypes.data, nblk, nchan,
                                                       None if pin is None else pin.ctypes.data, out.ctypes.data))
        return out

    def replay_device(self, dst_ptr=0, stream=0, kernel_mask=15):
        self._check(lib().gpsb200_replay_device(self._h, C.c_void_p(dst_ptr), C.c_void_p(stream), kernel_mask))
