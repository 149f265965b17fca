#!/usr/bin/env python3
"""Carrier NCO modes side by side: the FP64 carrier (the reference as shipped) against the U32 carrier (the reference
built without FLOAT_CARR_PHASE, gps.h:17) on bench.py's configs[2] workload -- 2999 blocks (300 s), int8, synthetic
parameters of bench.py's seed -- at 32 and at 12 channels, in ONE process, the two modes alternating step by step.

One JSON line per (mode, channels):
  ms_per_step     whole path per step: CUDA events on the launching stream around gpsb200_synth_blocks_device (host
                  records, parameters up, every kernel of the call), as bench.py's `value`
  kernels_ms      per kernel, replayed on the resident state of the last step (gpsb200_replay_device), CUDA events
  launches        kernels launched by one call (stats)
  synth_GBps      algorithmic bytes of the synthesis kernel (2 B per complex sample, int8) over its replayed time
  gpu, power_limit_w   the card and its power limit, read in the same run
Usage: python tools/bench_carrier_nco.py [--steps K] [--warmup W] [--out FILE]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
gps = importlib.import_module("multi-sdr-gps-sim_b200")

NBLK = 2999


def power_limit_w():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def workload(nchan, mode):
    ch, nav = gps.synthetic_chans(NBLK, nchan, seed=2024)
    if mode == "u32":                  # the same start phases as u32 accumulators
        ch["carr_phase"][0] = np.floor(ch["carr_phase"][0] * 4294967296.0)
    return ch, nav


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_carrier_nco: no CUDA device")
    dev_name, plim = torch.cuda.get_device_name(0), power_limit_w()
    lines = []
    for nchan in (32, 12):
        runs = {}
        for mode in ("fp64", "u32"):
            ch, nav = workload(nchan, mode)
            ctx = gps.Context(nchan, NBLK, carrier=mode)
            ctx.set_nav_frames(nav)
            out = torch.empty(NBLK * gps.BLOCK_ELEMS, dtype=torch.int8, device="cuda")
            runs[mode] = dict(ctx=ctx, ch=ch, out=out, ms=[], launches=0, host_chain_ms=0.0)
        stream = torch.cuda.Stream()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def step(r):
            torch.cuda.synchronize()
            ev0.record(stream)
            _, st = r["ctx"].synth_blocks_device(r["ch"], gps.SC08, r["out"].data_ptr(), stream.cuda_stream, want_stats=True)
            ev1.record(stream)
            stream.synchronize()
            return ev0.elapsed_time(ev1), st

        for _ in range(args.warmup):
            for mode in ("fp64", "u32"):
                step(runs[mode])
        for _ in range(args.steps):                          # alternating, so that both modes see the same box state
            for mode in ("fp64", "u32"):
                r = runs[mode]
                ms, st = step(r)
                r["ms"].append(ms)
                r["launches"] = int(st.launches)
                r["host_chain_ms"] += st.host_chain_ms / args.steps
        for mode in ("fp64", "u32"):
            r = runs[mode]
            ctx, sh, ptr = r["ctx"], stream.cuda_stream, r["out"].data_ptr()
            kev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            acc = [0.0] * 4
            reps = 3
            for _ in range(reps):
                kev[0].record(stream)
                for j, mask in enumerate((8, 4, 1, 2)):          # tables, probes + chaining, checkpoints, synthesis
                    ctx.replay_device(ptr, sh, mask)
                    kev[j + 1].record(stream)
                stream.synchronize()
                for j in range(4):
                    acc[j] += kev[j].elapsed_time(kev[j + 1]) / reps
            ms = np.array(r["ms"])
            kname = ctx.synth_kernel_name(nchan)
            line = dict(mode=mode, channels=nchan, blocks=NBLK, sample_size=1,
                        ms_per_step=round(float(ms.mean()), 3), ms_min=round(float(ms.min()), 3),
                        ms_max=round(float(ms.max()), 3), steps=args.steps,
                        kernels_ms={"k_tables": round(acc[0], 3), "k_probe+k_chain": round(acc[1], 3),
                                    "k_checkpoints": round(acc[2], 3), kname: round(acc[3], 3)},
                        synth_kernel=kname, launches=r["launches"], host_chain_ms=round(r["host_chain_ms"], 3),
                        synth_GBps=round(NBLK * gps.BLOCK_SAMPLES * 2 / (acc[3] * 1e-3) / 1e9, 1),
                        gpu=dev_name, power_limit_w=plim)
            print(json.dumps(line), flush=True)
            lines.append(line)
            ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
