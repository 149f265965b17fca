#!/usr/bin/env python3
"""bench.py -- IQ Msamples/s of the GPS L1 C/A synthesis hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--chan 32|12] [--iq16] [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input: the
300 s, 32-channel, int8 scenario of BASELINE.json configs[2] (2999 blocks of 0.1 s =
899.7 Msamples) per GPU. With N ranks the stream is N x 300 s long and time-sliced:
rank r synthesizes blocks [r*2999, (r+1)*2999) (weak scaling, no data-path collective).

  value  : whole-job Msamples/s of the WHOLE path per step, output left in an HBM buffer: host records and
           start-phase guesses, parameters up, carrier tables, block probes, span chaining, (N > 1: hand-over
           of the chain state over NCCL), host scan, run checkpoints + self-check, per-sample synthesis.
           CUDA events on the launching stream around all steps, max over ranks.
  e2e    : the same metric through the blocking C-ABI call with HOST buffers (N = 1: gpsb200_synth_blocks;
           N > 1: the three-step slice call): everything above plus the download of the int8/int16 stream
           into pinned memory inside the timed region.
  roofline: the synthesis kernel (k_synth_lanes, or k_synth when that does not apply) against the measured
           HBM copy peak; algorithmic bytes = 2 B per complex sample (int8 I+Q) written, nothing else
           counted (SURVEY.md section 8d).
  cpu_baseline / --impl reference: the reference's own producer loop (oracle/_ref/ref_run*,
           the unmodified gps.c behind a null sink) on this box's host cores.
  --dump-outputs DIR: after the timed steps, what the last one computed (see dump_outputs), so that two builds
           can be compared output for output; the inputs are seeded and identical from run to run.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# dram__bytes_read.sum + dram__bytes_write.sum (MB) of one 600-block int8 launch, by (kernel, more than 16 channels)
NCU_DRAM_MB = {("k_synth", True): 98.34 + 303.58, ("k_synth_lanes", True): 98.39 + 319.31, ("k_synth_lanes", False): 61.84 + 317.22}
BLOCKS_300S = 2999            # -d 300 -> round(10*300) - 1 blocks (gps.c:2703)
SAMPLES_PER_BLOCK = 300000
DUMP_BLOCKS = 16              # sampled blocks of --dump-outputs: at most 18 x 600000 float32 = 43.2 MB


def note(msg):
    """Progress line on stderr, flushed: if the box is lost mid-run the record still shows how far we got."""
    sys.stderr.write("[bench %s rank %s] %s\n" % (time.strftime("%H:%M:%S"), os.environ.get("RANK", "0"), msg))
    sys.stderr.flush()


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.

    NVML in-process every 5 ms (the timed region of the resident run is ~20 ms per step, far
    shorter than one `nvidia-smi` start-up); `nvidia-smi -lms` is the fallback when NVML cannot
    be loaded. Started before the warm-up steps so that it is running when the timed region opens;
    only samples whose time stamp falls inside the region are reported."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, uuid=None):
        self.rows = []            # (time, sm_mhz, set(reasons))
        self.max_mhz = None
        self.mode = None
        self.proc = None
        self._stop = threading.Event()
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            if uuid:
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
                except Exception:
                    h = None
            if h is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [v for v in vis.split(",") if v.strip().isdigit()]
                h = nv.nvmlDeviceGetHandleByIndex(int(ids[index]) if index < len(ids) else index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.nv, self.h, self.mode = nv, h, "nvml"
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.mode = "nvidia-smi"
            self.t = threading.Thread(target=self._pump_smi, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv, h = self.nv, self.h
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"),
                (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap"),
                (nv.nvmlClocksEventReasonHwPowerBrakeSlowdown, "hw_power_brake")]
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.rows.append((time.time(), mhz, {nm for b, nm in bits if mask & b}))
            except Exception:
                pass
            self._stop.wait(0.005)

    def _pump_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                mhz = float(r[0])
                self.max_mhz = max(self.max_mhz or 0.0, float(r[1]))
            except Exception:
                continue
            rs = {nm for k, nm in enumerate(names) if len(r) > 4 + k and r[4 + k].lower().startswith("active")}
            self.rows.append((time.time(), mhz, rs))

    def stop(self, t0, t1):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        if self.mode == "nvidia-smi":
            time.sleep(0.15)
            self.proc.terminate()
        self._stop.set()
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        where = "timed region"
        if not inside:                      # region shorter than the sampling period: nearest samples under load
            inside = [r for r in self.rows if t0 - 0.25 <= r[0] <= t1 + 0.05]
            where = "timed region +-0.25 s (warm-up load)"
        sm = [r[1] for r in inside]
        reasons = sorted(set().union(*[r[2] for r in inside])) if inside else []
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside), "source": self.mode, "window": where}


def host_cpus():
    """CPUs this process may really use: the cgroup quota when there is one, else the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, n)


def ref_binary(nchan, fast=False):
    name = "ref_run%d%s" % (32 if nchan > 12 else 12, "_fast" if fast else "")
    p = os.path.join(ROOT, "oracle", "_ref", name)
    return p if os.path.exists(p) else None


def run_reference_cpu(nchan, seconds, procs, fast=False):
    """Run `procs` independent copies of the reference producer (unmodified gps.c, null sink)
    on `seconds` of the sky-N static scenario. -> (Msamples/s aggregate, per-process list, wall)."""
    exe = ref_binary(nchan, fast)
    if exe is None:
        return None
    with tempfile.TemporaryDirectory() as td:
        nav = os.path.join(td, "sky.nav")
        subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "gen_rinex.py"),
                               "--nsat", str(32 if nchan > 12 else 12), "--out", nav])
        cmd = [exe, "-e", nav, "-l", "35.681298,139.766247,10.0", "-d", str(seconds), "-s", "2024/01/07,02:00:00"]
        t0 = time.time()
        ps = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, cwd=td)
              for _ in range(procs)]
        outs = [p.communicate()[0] for p in ps]
        wall = time.time() - t0
    per, samples = [], 0
    for o in outs:
        try:
            j = json.loads(o.strip().splitlines()[-1])
            per.append(j["samples"] / j["producer_seconds"] / 1e6)
            samples += j["samples"]
        except Exception:
            pass
    if not per:
        return None
    # aggregate = samples produced by all processes / the longest producer time (they run concurrently)
    agg = samples / max(s for s in [json.loads(o.strip().splitlines()[-1])["producer_seconds"] for o in outs]) / 1e6
    return agg, per, wall


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    nchan = args.chan
    procs = min(host_cpus(), 32)              # one copy per usable host core, never more than 32
    secs = 3.0 if nchan > 12 else 6.0         # 29 / 59 blocks per copy and step: ~2 s of CPU per step
    vals = []
    t_arm0 = time.time()
    warm = min(args.warmup, 2)                # CPU code has nothing to warm beyond the page cache
    for i in range(warm + args.steps):
        note("reference arm: step %d/%d, %d copies x %.0f s of signal" % (i + 1, warm + args.steps, procs, secs))
        r = run_reference_cpu(nchan, secs, procs)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_run* not built"}))
            return 0
        if i >= warm:
            vals.append(r)
        if time.time() - t_arm0 > 150.0 and len(vals) >= 2:     # bounded: the whole arm ends within a few minutes
            note("reference arm: time budget reached after %d timed steps" % len(vals))
            break
    agg = statistics.mean(v[0] for v in vals)
    single = statistics.mean(statistics.mean(v[1]) for v in vals)
    nblk = int(round(secs * 10)) - 1
    sample = ("%d concurrent copies of the reference producer (unmodified gps.c, -std=c11 -Og as shipped, null sink), "
              "each %d blocks (%.1f s of signal) of the sky-%d static scenario; the reference itself has one producer "
              "thread (%.2f Msps per copy)") % (procs, nblk, secs, 32 if nchan > 12 else 12, single)
    line = {
        "impl": "reference", "metric": "IQ Msamples/s", "value": round(agg, 3), "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": len(vals), "warmup": warm,
        "ms_per_step": round(1e3 * statistics.mean(v[2] for v in vals), 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 NCO / int32 accumulate / int8 out", "data": "synthetic",
        "config": workload_config(nchan, args.iq16, args.gpus, BLOCKS_300S if args.gpus == 1 else 35999,
                                         BLOCKS_300S if args.gpus == 1 else -(-35999 // args.gpus)),
        "cpu_baseline": {"value": round(agg, 3), "unit": "Msamples/s", "cores": procs, "kind": "reference",
                         "sample": sample, "single_thread_value": round(single, 3)},
        "e2e": {"value": round(agg, 3), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def workload_config(nchan, iq16, gpus, stream_blocks, per_rank_blocks):
    secs = (stream_blocks + 1) / 10.0
    return {"workload": "%d-channel synthetic constellation, %s, ONE %.0f s stream (%d blocks x 300000 samples), 3.0 Msps, "
                        "time-sliced %d-way (%s)" % (nchan, "int16" if iq16 else "int8", secs, stream_blocks, gpus,
                                                     "BASELINE configs[2]" if gpus == 1 and stream_blocks == BLOCKS_300S
                                                     else "BASELINE configs[4]" if stream_blocks == BLOCKS_3600S else "custom"),
            "channels": nchan, "stream_blocks": stream_blocks, "blocks_per_gpu": per_rank_blocks,
            "sample_format": "int16" if iq16 else "int8",
            "parallelism": "time-slice x%d; NCCL only for the hand-over of the slices' carrier-chain state "
                           "(guessed, then exact phases, rank to rank: send/recv); no data-path collective" % gpus,
            "l2": "output %.2f GB + checkpoints per rank and step >> 126 MB L2 (no flush needed)" % (
                per_rank_blocks * 600000 * (2 if iq16 else 1) / 1e9)}


BLOCKS_3600S = 35999          # BASELINE configs[4]: -d 3600


def dump_outputs(dirname, out_dev, block_elems, phases, prefix=""):
    """Write what a caller of the timed path receives from one step, as .npy:
      carrier_phase.npy  float64 [channels]: the exact carrier phases at the end of the slice (all of them)
      iq_sample.npy      float32 [n, block_elems]: whole blocks of the int8/int16 IQ stream (interleaved I, Q),
                         a fixed, seeded sample of them (the stream is 1.8 GB for the default workload)
      iq_sample_block.npy float64 [n]: the indices of those blocks in the slice (first and last always included)"""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    nblk = out_dev.numel() // block_elems
    pick = np.random.default_rng(0).choice(nblk, size=min(DUMP_BLOCKS, nblk), replace=False)
    pick = np.unique(np.concatenate([[0, nblk - 1], pick]))
    iq = out_dev.view(nblk, block_elems)[torch.from_numpy(pick).to(out_dev.device)].float().cpu().numpy()
    np.save(os.path.join(dirname, prefix + "carrier_phase.npy"), np.asarray(phases, dtype=np.float64))
    np.save(os.path.join(dirname, prefix + "iq_sample.npy"), iq)
    np.save(os.path.join(dirname, prefix + "iq_sample_block.npy"), pick.astype(np.float64))


class HandOver:
    """The carrier-chain hand-over of a time-sliced stream over NCCL (include/gpsb200.h, "time-slice hand-over"):
    every step two small messages (32 satellite ids + 32 phases each) travel rank to rank with send/recv -- first the
    GUESSED state (closed-form links composed down the ranks, available before any GPU work), later the EXACT one.
    Nothing else crosses NVLink."""

    def __init__(self, gps, world, rank, nchan):
        import numpy as np
        import torch
        import torch.distributed as dist
        self.gps, self.world, self.rank, self.nchan = gps, world, rank, nchan
        self.np, self.torch, self.dist = np, torch, dist
        if world > 1:
            self.guess_in = torch.zeros(64, dtype=torch.float64, device="cuda")
            self.guess_out = torch.zeros(64, dtype=torch.float64, device="cuda")
            self.state_dev = torch.zeros(64, dtype=torch.float64, device="cuda")
            self.state_out = torch.zeros(64, dtype=torch.float64, device="cuda")

    def guessed_incoming(self, link):
        """The GUESSED state entering this rank's slice, passed down the ranks: receive the guess composed by the
        predecessors, apply the own slice's closed-form link (gpsb200_link_apply), send the result on. Only ranks
        r' < r matter to rank r, so nothing here makes an early rank wait for a late one: consecutive steps overlap
        across ranks like the stages of a pipeline. -> (prn, phase), (None, None) for rank 0."""
        if self.world == 1:
            return None, None
        np, gps = self.np, self.gps
        prn, ph = None, None
        if self.rank > 0:
            for w in self.dist.batch_isend_irecv([self.dist.P2POp(self.dist.irecv, self.guess_in, self.rank - 1)]):
                w.wait()
            v = self.guess_in.cpu().numpy()
            prn, ph = v[:32][:self.nchan].astype(np.int32), v[32:][:self.nchan].copy()
        if self.rank + 1 < self.world:
            pn, xn = gps.link_apply(link, self.nchan, prn, ph)
            v = np.zeros(64)
            v[:self.nchan] = pn
            v[32:32 + self.nchan] = xn
            self.guess_out.copy_(self.torch.from_numpy(v))
            for w in self.dist.batch_isend_irecv([self.dist.P2POp(self.dist.isend, self.guess_out, self.rank + 1)]):
                w.wait()
        return prn, ph

    def recv_exact(self):
        if self.rank == 0:
            return None, None
        for w in self.dist.batch_isend_irecv([self.dist.P2POp(self.dist.irecv, self.state_dev, self.rank - 1)]):
            w.wait()
        v = self.state_dev.cpu().numpy()
        return v[:32][:self.nchan].astype(self.np.int32), v[32:][:self.nchan].copy()

    def send_exact(self, prn, ph):
        if self.rank + 1 >= self.world:
            return
        np = self.np
        v = np.zeros(64)
        v[:self.nchan] = prn
        v[32:32 + self.nchan] = ph
        self.state_out.copy_(self.torch.from_numpy(v))
        for w in self.dist.batch_isend_irecv([self.dist.P2POp(self.dist.isend, self.state_out, self.rank + 1)]):
            w.wait()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpsb200")
    ap.add_argument("--chan", type=int, default=32)
    ap.add_argument("--iq16", action="store_true")
    ap.add_argument("--stream-seconds", type=float, default=0.0,
                    help="length of the ONE stream all ranks share (default: 300 s = configs[2] on 1 GPU, 3600 s = configs[4] on N > 1)")
    ap.add_argument("--blocks", type=int, default=0, help="stream length in blocks (overrides --stream-seconds)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--gather", action="store_true", help="also time an NCCL all-gather of the finished slices")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not bind the rank to its GPU's NUMA node (A/B)")
    ap.add_argument("--run-samples", type=int, default=0, help="device work unit (0 = library default)")
    ap.add_argument("--depth", type=int, default=2, help="contexts used alternately by consecutive steps (1: no overlap)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/*.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    gps = importlib.import_module("multi-sdr-gps-sim_b200")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: gpsb200 has no CPU fallback")
    torch.cuda.set_device(local)
    # the rank's threads and its page-locked result buffer go to the NUMA node of its GPU (library helper)
    numa_node = None if args.no_numa_bind else gps.bind_numa(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # no "NCCL version ..." banner on stdout: ONE JSON line
        # high-priority NCCL streams: the hand-over messages are tiny kernels that must not wait behind walk kernels
        opts = None
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            opts = None
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local), pg_options=opts)
        except TypeError:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    nchan = args.chan
    if args.blocks > 0:
        total_blocks = args.blocks
    elif args.stream_seconds > 0:
        total_blocks = int(args.stream_seconds * 10 + 0.5) - 1
    else:
        total_blocks = BLOCKS_300S if world == 1 else BLOCKS_3600S
    lo, hi = gps.sharding.slice_bounds(total_blocks, world, rank)
    nblk = hi - lo
    max_nblk = gps.sharding.slice_bounds(total_blocks, world, 0)[1]
    note("device %d of %d ranks: blocks [%d, %d) of a %d-block stream, %d channels" % (local, world, lo, hi, total_blocks, nchan))
    ss = gps.SC16 if args.iq16 else gps.SC08
    bytes_per_sample = 4 if args.iq16 else 2
    # this rank's slice of ONE continuous scenario; nothing about the blocks before it is precomputed
    chans, nav = gps.synthetic_chans(nblk, nchan, seed=2024, block0=lo)
    # host workers per rank: the ranks' host phases are staggered (each rank scans when its predecessor has handed over),
    # so a rank may use more than its even share of the CPUs
    host_threads = max(2, min(16, host_cpus() // max(1, (world + 1) // 2)))
    # Double buffering (--depth 2): consecutive steps alternate between two contexts with their own streams and
    # output buffers, so that the speculative pre-phase of step k+1 (host records, probes, span chaining) runs while
    # step k is still being synthesized -- what a streaming producer of successive stream chunks does. A step is still
    # ONE pass of the whole path over one batch; K steps are timed from a common start to the completion of the last.
    depth = max(1, args.depth)
    ctxs, outs, streams = [], [], []
    for _ in range(depth):
        c = gps.Context(nchan, max_nblk, device=local, max_nav_frames=1, host_threads=host_threads,
                        run_samples=args.run_samples)
        c.set_nav_frames(nav)
        ctxs.append(c)
        outs.append(torch.empty(nblk * gps.BLOCK_ELEMS, dtype=torch.int16 if args.iq16 else torch.int8, device="cuda"))
        # dedicated (non-default) streams: handle 0 would mean "the context's own stream" to the C ABI
        streams.append(torch.cuda.Stream())
    ctx, out_dev, stream = ctxs[0], outs[0], streams[0]
    sh = stream.cuda_stream
    assert sh != 0
    slot = [0]            # which context / stream / output buffer the next step uses
    ho = HandOver(gps, world, rank, nchan)
    step_trace = []       # BENCH_TRACE=1: per step [prepare, links all-gather, probe, recv exact, finish(+send)] ms, host share

    def one_step(dst_ptr=0, dst_host=None):
        """One pass of the whole hot path over this rank's slice: host records, parameters up, carrier tables, block
        probes, span chaining, hand-over, host scan, run checkpoints (+ self-check), synthesis. -> Stats"""
        ctx, sh = ctxs[slot[0]], streams[slot[0]].cuda_stream
        if dst_ptr == "slot":
            dst_ptr = outs[slot[0]].data_ptr()
        if world == 1 and dst_host is None:
            # one GPU: the public device-destination call (the same steps, pipelined segment by segment; it returns
            # once everything is enqueued and the chain self-check of the whole call has been read)
            ph, st1 = ctx.synth_blocks_device(chans, ss, dst_ptr, stream=sh, want_stats=True)
            return st1, ph
        tr = [time.perf_counter()]
        link = ctx.slice_prepare(chans, ss, dst_ptr, stream=sh, dst_host=dst_host)
        tr.append(time.perf_counter())
        gprn, gph = ho.guessed_incoming(link) if world > 1 else (None, None)
        tr.append(time.perf_counter())
        # eager on every rank of a multi-GPU run: a successor waits for the outgoing state, and the last rank has to wait
        # for its incoming state anyway -- time in which all of its probes complete
        ctx.slice_probe(gprn, gph, eager=world > 1)
        tr.append(time.perf_counter())
        prn_in, ph_in = ho.recv_exact() if world > 1 else (None, None)
        tr.append(time.perf_counter())
        # the exact outgoing state goes to the successor from inside the call, BEFORE the long kernels are enqueued (an
        # NCCL send is a kernel too and would otherwise wait behind this rank's own synthesis)
        prn_out, ph_out, st = ctx.slice_finish(prn_in, ph_in, want_stats=True,
                                               handoff=ho.send_exact if rank + 1 < world else None)
        tr.append(time.perf_counter())
        if os.environ.get("BENCH_TRACE"):
            step_trace.append([round((b - a) * 1e3, 3) for a, b in zip(tr[:-1], tr[1:])] + [round(st.host_chain_ms, 3)])
        return st, ph_out

    # ---- value: the whole path, parameters in host memory (6 MB), result left in HBM ---------------------
    note("value leg: first full pass")
    def step_wait(k=None):
        """Wait for the step that last used context k (default: the current slot)."""
        k = slot[0] if k is None else k
        if world == 1:
            streams[k].synchronize()
        else:
            ctxs[k].slice_wait()      # completion + verdict of the device self-check

    for k in range(depth):            # first full pass on every context
        slot[0] = k
        st, _ = one_step("slot")
        step_wait()
    slot[0] = 0
    sampler = None
    if rank == 0:
        uuid = getattr(torch.cuda.get_device_properties(local), "uuid", None)
        sampler = ClockSampler(local, uuid)
    note("value leg: %d warm-up + %d timed steps" % (args.warmup, args.steps))
    for _ in range(args.warmup):
        one_step("slot")
        step_wait()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern = {"k_probe_chain_ms": 0.0, "k_checkpoints_ms": 0.0, "k_synth_ms": 0.0, "host_chain_ms": 0.0}
    fallbacks = 0
    launches = 0
    t_wall0 = time.time()
    tstream = torch.cuda.Stream()      # timing events: the device is idle at ev0 (barrier) and at ev1 (synchronize)
    ev0.record(tstream)
    busy = [False] * depth
    for i in range(args.steps):
        slot[0] = i % depth
        if busy[slot[0]]:
            step_wait()                                       # this context's previous step: its buffers are reused now
        st, ph_last = one_step("slot")
        busy[slot[0]] = True
        kern["host_chain_ms"] += st.host_chain_ms
        fallbacks += st.chain_fallbacks
        launches += int(st.launches)
    for k in range(depth):
        if busy[k]:
            step_wait(k)
    torch.cuda.synchronize()
    ev1.record(tstream)
    torch.cuda.synchronize()
    barrier()
    slot[0] = (args.steps - 1) % depth                        # the context of the last step: its state is replayed below
    ctx, out_dev, stream = ctxs[slot[0]], outs[slot[0]], streams[slot[0]]
    sh = stream.cuda_stream
    t_wall1 = time.time()
    total_ms = ev0.elapsed_time(ev1)
    if os.environ.get("BENCH_TRACE") and step_trace:
        note("step phases [prepare, links, probe, recv, finish+send | host_chain] ms: %s" % step_trace[-3:])
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if args.dump_outputs:                                     # before the replays below rewrite the buffer
        dump_outputs(args.dump_outputs, out_dev, gps.BLOCK_ELEMS, ph_last, "rank%d_" % rank if world > 1 else "")
        note("outputs of the last timed step written to %s" % args.dump_outputs)
    total_ms = max_over_ranks(total_ms)
    ms_per_step = total_ms / args.steps
    samples_all = total_blocks * SAMPLES_PER_BLOCK
    value = samples_all / (ms_per_step * 1e-3) / 1e6
    # per-kernel times: the same kernels replayed on the resident state of the last step, CUDA events on the
    # launching stream (the timed steps above interleave host work, so they are bracketed separately here)
    kev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    reps = max(3, min(args.steps, 5))
    acc = [0.0] * 4
    for _ in range(reps):
        kev[0].record(stream)
        ctx.replay_device(out_dev.data_ptr(), sh, 8)      # gain-scaled carrier tables of every block
        kev[1].record(stream)
        ctx.replay_device(out_dev.data_ptr(), sh, 4)      # speculative carrier probes + span chaining
        kev[2].record(stream)
        ctx.replay_device(out_dev.data_ptr(), sh, 1)      # run checkpoints (exact NCO fast-forward) + chain self-check
        kev[3].record(stream)
        ctx.replay_device(out_dev.data_ptr(), sh, 2)      # per-sample synthesis
        kev[4].record(stream)
        stream.synchronize()
        for j in range(4):
            acc[j] += kev[j].elapsed_time(kev[j + 1]) / reps
    tb_ms, pr_ms, ck_ms, syn_ms = acc

    # ---- end to end: the same path with a HOST destination (pinned), downloads overlapped ----------------
    e2e, e2e_err = None, None
    if not args.no_e2e:
        note("value leg done: %.3f ms per step; end-to-end leg (pinned host buffer %.2f GB)" % (
            ms_per_step, nblk * gps.BLOCK_ELEMS * (2 if args.iq16 else 1) / 1e9))
        try:
            out_host = torch.empty(nblk * gps.BLOCK_ELEMS, dtype=torch.int16 if args.iq16 else torch.int8, pin_memory=True)
            out_np = out_host.numpy()
            e2e_steps = args.steps

            def e2e_step():
                if world == 1:          # the blocking public call: segmented pipeline, chain resolution of later
                    _, _, s2 = ctx.synth_blocks(chans, ss, out=out_np, want_stats=True)   # segments under the downloads
                    return s2
                s2, _ = one_step(0, out_np)     # N > 1: the three-step call with the hand-over, host destination
                ctx.slice_wait()
                return s2

            e2e_step()
            barrier()
            t0 = time.perf_counter()
            e2e_each = []
            for _ in range(e2e_steps):
                t1 = time.perf_counter()
                st2 = e2e_step()
                e2e_each.append(time.perf_counter() - t1)
            torch.cuda.synchronize()
            e2e_s = (time.perf_counter() - t0) / e2e_steps
            e2e_s = max_over_ranks(e2e_s)
            e2e_value = samples_all / e2e_s / 1e6
            # result check: the end-to-end output equals the resident-output run (same bytes)
            same = bool(torch.equal(out_host.cuda(), out_dev))
            same = bool(max_over_ranks(0.0 if same else 1.0) == 0.0)
            e2e = {"value": round(e2e_value, 1), "unit": "Msamples/s",
                   "h2d_bytes_per_step": int(st2.h2d_bytes) * world, "d2h_bytes_per_step": int(st2.d2h_bytes) * world,
                   "ms_per_step": round(e2e_s * 1e3, 2), "steps": e2e_steps,
                   "ms_best_step_rank0": round(min(e2e_each) * 1e3, 2), "host_chain_ms": round(st2.host_chain_ms, 2),
                   "chain_fallbacks": int(st2.chain_fallbacks), "kernel_launches_per_step": int(st2.launches),
                   "host_threads": host_threads, "numa_node": numa_node,
                   "timing": "wall clock around the call (hand-over included), max over ranks",
                   "output_equals_resident_run": same}
            del out_host, out_np
        except Exception as ex:                      # the line is still printed, with the reason
            e2e_err = "%s: %s" % (type(ex).__name__, ex)
            note("end-to-end leg failed: " + e2e_err)

    gather_ms = None
    if args.gather and world > 1 and total_blocks % world == 0:
        full = torch.empty(world * out_dev.numel(), dtype=out_dev.dtype, device="cuda")
        dist.all_gather_into_tensor(full, out_dev)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        dist.all_gather_into_tensor(full, out_dev)
        g1.record()
        barrier()
        gather_ms = max_over_ranks(g0.elapsed_time(g1))

    if rank == 0:
        peak, peak_src = read_peaks()
        alg_bytes = nblk * SAMPLES_PER_BLOCK * bytes_per_sample        # one k_synth launch of this rank
        achieved = alg_bytes / (syn_ms * 1e-3) / 1e9
        synth_kernel = ctxs[0].synth_kernel_name(nchan)
        line = {
            "metric": "IQ Msamples/s", "value": round(value, 1), "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3),
            "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
            "dtype": "f64 NCO / int32 accumulate / %s out" % ("int16" if args.iq16 else "int8"),
            "data": "synthetic", "config": workload_config(nchan, args.iq16, world, total_blocks, nblk),
            "clocks": clocks, "gpu_launches": launches,
            "pipeline_depth": depth,
            "timed_region": "per step the WHOLE path of the rank's slice: host records + guesses, 6 MB of parameters up, "
                            "carrier tables, block probes, span chaining, hand-over of the chain state (N > 1: NCCL "
                            "all-gather + send/recv), host scan, run checkpoints + self-check, synthesis into HBM",
            "value_kernels_only": round(samples_all / world / ((tb_ms + pr_ms + ck_ms + syn_ms) * 1e-3) / 1e6 * world, 1)
            if world == 1 else None,
            "kernels": {"k_tables_ms": round(tb_ms, 3), "k_probe_chain_ms": round(pr_ms, 3), "k_checkpoints_ms": round(ck_ms, 3),
                        "k_synth_ms": round(syn_ms, 3), "host_chain_ms_per_step": round(kern["host_chain_ms"] / args.steps, 3),
                        "chain_fallback_blocks_per_step": fallbacks / args.steps,
                        "note": "kernels replayed back to back on the last step's resident state, CUDA events on the launching stream"},
            "roofline": {"bound": "hbm", "kernel": synth_kernel, "achieved": round(achieved, 1), "peak": peak,
                         "unit": "GB/s", "frac": round(achieved / peak, 4),
                         # ncu --set full (profiles/r2_ncu_metrics.csv): dram read+write of one 600-block int8 launch
                         # (360 MB of algorithmic bytes), scaled to this launch
                         "traffic": (int(alg_bytes * NCU_DRAM_MB.get((synth_kernel, nchan > 16), 0.0) / 360.0) or None)
                         if not args.iq16 else None,
                         "peak_source": peak_src,
                         "note": "the kernel is bound by integer issue slots and shared-memory look-ups, not by HBM; see DESIGN.md and profiles/"},
            "e2e": e2e if e2e is not None else {"value": None, "unit": "Msamples/s", "error": e2e_err or "skipped (--no-e2e)"},
        }
        if gather_ms is not None:
            line["nccl_all_gather_ms"] = round(gather_ms, 3)
        if not args.no_cpu_baseline and world == 1:
            note("cpu_baseline leg: one copy of the reference producer")
            try:
                r = run_reference_cpu(nchan, 10.0 if nchan <= 12 else 5.0, 1)
            except Exception as ex:
                r = None
                line["cpu_baseline"] = {"value": None, "error": "%s: %s" % (type(ex).__name__, ex)}
            if r is not None:
                line["cpu_baseline"] = {
                    "value": round(r[0], 3), "unit": "Msamples/s", "cores": 1, "kind": "reference",
                    "sample": "reference producer loop (unmodified gps.c, -std=c11 -Og as shipped, null sink), "
                              "%d blocks of the sky-%d static scenario, one producer thread (all the reference has)"
                              % (99 if nchan <= 12 else 49, 32 if nchan > 12 else 12)}
        print(json.dumps(line))
    for c in ctxs:
        c.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
