"""gpsb200: B200-native GPS L1 C/A baseband synthesis (hot path of multi-sdr-gps-sim).

The product is libgpsb200.so (CUDA kernels for sm_100a behind the C ABI of
include/gpsb200.h). This package is only the host-side convenience layer used by
the tests and bench.py: ctypes bindings that mirror the C ABI one to one.
Import it with importlib (the directory name is not a Python identifier):

    gps = importlib.import_module("multi-sdr-gps-sim_b200")
"""
from .api import (  # noqa: F401
    BLOCK_ELEMS, BLOCK_SAMPLES, SC08, SC16, Chan, Config, Context, GpsB200Error, Stats,
    bind_numa, carrier_advance, span_chain_host, lanes_model_block, link_apply, slice_link_host, SliceLink, carrier_chain, codegen, scenario, lib, lib_path, CHAN_DTYPE,
    CARRIER_FP64, CARRIER_U32, carrier_advance_u32,
)
from .synthetic import synthetic_chans  # noqa: F401,E402
from . import sharding  # noqa: F401,E402
