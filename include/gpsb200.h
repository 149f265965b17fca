/* gpsb200 -- B200-native GPS L1 C/A baseband synthesis, C ABI.
 *
 * Drop-in for the sample loop of the reference's producer thread
 * (Mictronics/multi-sdr-gps-sim, gps_thread_ep): everything between the 10 Hz
 * channel update (gps.c:2731-2765) and fifo_enqueue (gps.c:2860) -- i.e.
 * gps.c:2767-2857 -- runs as sm_100a CUDA kernels behind these entry points.
 * Plain C types only; no C++/torch types cross this boundary.
 *
 * The second half of this header re-declares, unchanged, the FIFO / sink API of
 * the reference (fifo.h:19-62, sdr.h:18-39 constants) which libgpsb200.so also
 * exports (pinned host buffers, fixed tail handling) so that the reference's
 * consumers (sdr_iqfile.c:22-55, sdr_hackrf.c:236-248, sdr_pluto.c:45-94) work
 * unmodified against it.
 */
#ifndef GPSB200_H
#define GPSB200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- constants of the reference (sdr.h:21-34, gps.h:36-57) ------------------ */
#define GPSB200_SAMPLERATE        3000000           /* TX_SAMPLERATE, sdr.h:21 */
#define GPSB200_BLOCK_SAMPLES     300000            /* NUM_IQ_SAMPLES, sdr.h:26 */
#define GPSB200_BLOCK_ELEMS       600000            /* IQ_BUFFER_SIZE, sdr.h:29 (I and Q count separately) */
#define GPSB200_MAX_CHAN          32                /* reference ships MAX_CHAN 12 (gps.h:36); 32 = all PRNs */
#define GPSB200_NAV_WORDS         60                /* N_DWRD, gps.h:52 */
#define GPSB200_CA_LEN            1023              /* CA_SEQ_LEN, gps.h:57 */
#define GPSB200_SC08              1                 /* gps-sim.h:27 */
#define GPSB200_SC16              2                 /* gps-sim.h:28 */
#define GPSB200_HACKRF_BUFFER     262144            /* HACKRF_TRANSFER_BUFFER_SIZE, sdr.h:34 */

/* ---- error codes ------------------------------------------------------------ */
enum {
    GPSB200_OK = 0,
    GPSB200_ERR_ARG = -1,        /* bad argument (NULL, count, sample size, prn, NAV index) */
    GPSB200_ERR_CUDA = -2,       /* CUDA runtime error; text via gpsb200_last_error() */
    GPSB200_ERR_RANGE = -3,      /* sum of channel amplitudes would overflow the int16 I/Q the reference stores */
    GPSB200_ERR_NOMEM = -4,
    GPSB200_ERR_INTERNAL = -5    /* device self-check failed (would mean a bug; never returns wrong samples silently) */
};

/* ---- carrier NCO of the reference build being replaced (gps.h:17) -------------------------------------------
 * GPSB200_CARRIER_FP64 (default): `#define FLOAT_CARR_PHASE` present, as shipped: double carr_phase in [0,1),
 *     carr_phase += f_carr * delt with a wrap per sample, table index floor(carr_phase * 512) (gps.c:2775, 2821-2826).
 * GPSB200_CARRIER_U32: the define absent: unsigned int carr_phase, carr_phasestep = (int) round(512.0 * 65536.0 *
 *     f_carr * delt) per block (gps.c:2745-2747), table index (carr_phase >> 16) & 511, carr_phase += carr_phasestep
 *     modulo 2^32 per sample (gps.c:2777, 2828), allocation phase (unsigned int) (512.0 * 65536.0 * frac(phase_ini))
 *     (gps.c:2212-2213). In a U32 context every carrier phase the API takes or returns (gpsb200_chan_t.carr_phase,
 *     carr_phase_out, the slice calls' phase_in / phase_out / phase_guess_in, gpsb200_carrier_chain_device) is that
 *     accumulator as an integer-valued double in [0, 2^32); any other value is GPSB200_ERR_ARG. The phase at any sample
 *     is then a closed form, so these contexts launch no carrier-chain kernels at all. */
#define GPSB200_CARRIER_FP64      0
#define GPSB200_CARRIER_U32       1

/* One channel for one 0.1 s block: the fields of the reference's channel_t
 * (gps.h:213-236) and gain[] (gps.c:2300) that the sample loop reads, as left by
 * computeCodePhase (gps.c:2033-2064) and the gain update (gps.c:2749-2763).
 * dataBit/codeCA are not passed: they are functions of (iword, ibit, NAV words)
 * and (code_phase, prn) respectively (gps.c:2059-2060). */
typedef struct gpsb200_chan {
    int32_t prn;          /* 1..32; <= 0: channel unused this block (gps.c:2772) */
    int32_t iword;        /* NAV word index 0..59  (gps.c:2052) */
    int32_t ibit;         /* bit in word 0..29     (gps.c:2055) */
    int32_t icode;        /* code period in bit 0..19 (gps.c:2058) */
    int32_t nav_frame;    /* which NAV frame (set of 60 words) this block uses, see gpsb200_set_nav */
    int32_t reserved;
    double f_carr;        /* Hz, Doppler (gps.c:2043); |f_carr| < 2.9 MHz */
    double f_code;        /* Hz (gps.c:2044); 0 < f_code <= 1.07 MHz */
    double carr_phase;    /* cycles in [0,1) (GPSB200_CARRIER_U32: the u32 accumulator, see above): used for the first block of a call and whenever prn differs
                             from the previous block's prn in the same slot (allocateChannel, gps.c:2203-2210);
                             otherwise the phase is carried from the previous block (gps.c:2821-2826) */
    double code_phase;    /* chips in [0,1023) (gps.c:2049) */
    double gain;          /* gps.c:2756 (x2 for Pluto, gps.c:2759-2763) */
} gpsb200_chan_t;         /* 64 bytes */

typedef struct gpsb200_config {
    int32_t device;            /* CUDA device ordinal */
    int32_t max_chan;          /* 1..32 */
    int32_t max_blocks;        /* largest nblk of one gpsb200_synth_* call */
    int32_t max_nav_frames;    /* NAV frames held at once (>= 1) */
    int32_t host_threads;      /* threads for the exact carrier-phase chain; 0 = auto */
    int32_t run_samples;       /* device work unit, divides 300000 and is a multiple of 32; 0 = default (2400) */
    int32_t carrier_nco;       /* GPSB200_CARRIER_FP64 (0) or GPSB200_CARRIER_U32. Added last in version 0.3: callers
                                  must be rebuilt against this header (the struct grew by 4 bytes) */
} gpsb200_config_t;

typedef struct gpsb200_ctx gpsb200_ctx_t;

/* Per-call statistics (filled when the pointer is not NULL). Times in milliseconds. */
typedef struct gpsb200_stats {
    double host_chain_ms;      /* host share of the carrier chain: start-phase guesses + fix-up scan */
    double h2d_ms, kernel_ms, d2h_ms;   /* kernel_ms: CUDA-event span of the call's stream (host-destination calls only);
                                           h2d_ms / d2h_ms: reserved, always 0 (transfers overlap the kernels) */
    double checkpoint_kernel_ms, synth_kernel_ms, probe_kernel_ms;
    int64_t h2d_bytes, d2h_bytes;
    int32_t launches;          /* kernels launched by this call */
    int32_t chain_fallbacks;   /* blocks the host had to walk sequentially (their block probe was unusable) */
} gpsb200_stats_t;

/* Threading: a context may be used by one thread at a time; different contexts (same or different devices)
 * may be used concurrently from different threads, every entry point selects the context's device itself.
 * The FIFO below is process-global with one producer and one consumer, as in the reference (fifo.c:21-29). */
int gpsb200_create(const gpsb200_config_t *cfg, gpsb200_ctx_t **out);
void gpsb200_destroy(gpsb200_ctx_t *ctx);
const char *gpsb200_last_error(const gpsb200_ctx_t *ctx);
const char *gpsb200_version(void);

/* Deployment helper, the counterpart of the reference's thread_to_core() (gps-sim.c:251-262, called by
 * gps_thread_ep, gps.c:2377): bind the CALLING thread (and every thread it creates afterwards: the
 * context's host workers, the iqfile writer) to the CPUs of the NUMA node the CUDA device `device`
 * hangs off, so that page-locked result buffers allocated afterwards (fifo_create, cudaHostAlloc) are
 * local to the GPU's PCIe root. Call before gpsb200_create / fifo_create. Returns the NUMA node (>= 0),
 * -1 when the platform reports none (nothing changed), or GPSB200_ERR_CUDA. */
int gpsb200_bind_numa(int device);

/* NAV words of one channel for one 30 s frame: channel_t.dwrd (gps.h:227) as
 * built by generateNavMsg (gps.c:2066-2140); only bits 29..0 are used
 * (gps.c:2812). Copied; may be updated between synth calls. */
int gpsb200_set_nav(gpsb200_ctx_t *ctx, int frame, int chan, const uint32_t dwrd[GPSB200_NAV_WORDS]);

/* Synthesize nblk consecutive 0.1 s blocks (replaces gps.c:2767-2857 nblk times).
 *   chans       [nblk][nchan], host memory; 1 <= nchan <= cfg.max_chan (slot c of a call is NAV row c of the context)
 *   sample_size GPSB200_SC08: dst is int8  I,Q interleaved, iq >> 4 with modulo-256 narrowing (gps.c:2844)
 *               GPSB200_SC16: dst is int16 I,Q interleaved (gps.c:2842)
 *   dst         host memory (pinned is faster), nblk * 600000 elements, block after block
 *   carr_phase_out  optional [nchan]: carrier phase after the last block (what the reference
 *               leaves in channel_t.carr_phase), to seed the next call
 * Blocking: returns when dst is complete. */
int gpsb200_synth_blocks(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan,
                         int sample_size, void *dst, double *carr_phase_out, gpsb200_stats_t *stats);

/* Same, but block b goes to its own host buffer dst_blocks[b] (600000 elements each) -- e.g. buffers handed out by
 * fifo_acquire(): the device->host copies land straight in iq->data8 / iq->data16 (SURVEY 8b ownership: the producer
 * owns a buffer between acquire and enqueue), no staging copy on the host. */
int gpsb200_synth_blocks_scatter(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan,
                                 int sample_size, void *const *dst_blocks, double *carr_phase_out,
                                 gpsb200_stats_t *stats);

/* Same, but the output stays in device memory (dst_device: device pointer with room for
 * nblk * 600000 elements) and the synthesis is only ENQUEUED on `stream` (a cudaStream_t,
 * 0 = the context's own stream) -- the caller synchronizes before reading dst_device. The call itself returns when
 * the speculative pre-phase (block probes, span chaining), the host scan and the run checkpoints are done and the
 * device self-check of the carrier chain has been read (a failed check returns GPSB200_ERR_INTERNAL, and nothing of the
 * call is left in flight); it never waits for the synthesis, with or without a stats request (stats then carry no
 * synthesis time). Used for kernel-resident consumers and by bench.py's one-GPU value leg. */
int gpsb200_synth_blocks_device(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan,
                                int sample_size, void *dst_device, void *stream,
                                double *carr_phase_out, gpsb200_stats_t *stats);

/* ---- time-slice hand-over (multi-GPU: rank r makes blocks [lo_r, hi_r) of ONE stream) -----------------
 * The only state a slice needs from the blocks before it is each slot's exact carrier phase (gps.c:2821-2826
 * never resets carr_phase). Its resolution is parallel in time (block probes on the GPU chained per span, then
 * one host step per span), so a rank can do almost all of it before the incoming phases exist. One device-path
 * call is therefore offered in three steps:
 *   1. gpsb200_slice_prepare  host records, parameters up, carrier tables; fills *link: how this slice maps an
 *                             incoming chain state to the (closed-form, GUESSED) outgoing one. Ranks exchange
 *                             their links and compose them with gpsb200_link_apply() to obtain good guesses of
 *                             their incoming state without any GPU work.
 *   2. gpsb200_slice_probe    incoming state as GUESSED (NULL: the slice starts the stream): speculative block
 *                             probes + span chaining are enqueued (all of them at once if `eager`).
 *   3. gpsb200_slice_finish   incoming state EXACT (prn_in/phase_in, from the previous rank's *_out; NULL: the
 *                             stream starts here): segment by segment, as soon as a segment's probes are done, the
 *                             host scan over its span summaries, its run checkpoints (with the device self-check) and
 *                             its synthesis are enqueued -- the synthesis of early segments overlaps the probes of
 *                             later ones. prn_out/phase_out (exact state after the slice) are valid on return --
 *                             BEFORE the synthesis has run -- and are what the next rank's gpsb200_slice_finish takes.
 *   4. gpsb200_slice_wait     blocks until the slice is complete and returns the verdict of the device self-check
 *                             (GPSB200_ERR_INTERNAL: the output must not be used).
 * A slot continues the incoming phase only when it still holds the same satellite (prn_in[c] == prn of its first
 * block, > 0); otherwise its first block takes carr_phase from chans, exactly as between the blocks of one call.
 * chans must stay valid until gpsb200_slice_prepare returns. gpsb200_synth_blocks_device == the three steps with
 * NULL incoming states. */
typedef struct gpsb200_slice_link {
    int32_t prn_first[GPSB200_MAX_CHAN];    /* satellite of each slot in the slice's first block (0: idle) */
    int32_t prn_last[GPSB200_MAX_CHAN];     /* ... in its last block */
    int32_t reset_inside[GPSB200_MAX_CHAN]; /* 1: the slot was (re)allocated or idle inside the slice: value is absolute */
    double first_phase[GPSB200_MAX_CHAN];   /* carr_phase of the first block (used when the slot does not continue) */
    double value[GPSB200_MAX_CHAN];         /* guessed phase after the slice (absolute), or the advance over the slice */
} gpsb200_slice_link_t;
/* dst_device and/or dst_host: with dst_host != NULL the synthesis is launched in chunks whose downloads into dst_host
 * (pinned memory) overlap later chunks, dst_device may then be NULL (a context-owned staging buffer is used);
 * gpsb200_slice_wait blocks until synthesis and downloads of the slice are complete and reports the self-check. */
int gpsb200_slice_prepare(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size,
                          void *dst_device, void *dst_host, void *stream, gpsb200_slice_link_t *link);
int gpsb200_slice_wait(gpsb200_ctx_t *ctx);
/* eager != 0: the speculative work of the WHOLE slice is submitted at once, ahead of everything else -- for a rank
 * whose successor waits for the outgoing state. eager == 0: only the first pipeline segment's; the others follow
 * segment by segment inside gpsb200_slice_finish, each behind the previous segment's synthesis (in whose shadow the
 * latency-bound walk kernels then run) and from guesses re-anchored on the exact state just resolved -- for the last
 * rank and for single-GPU use. */
int gpsb200_slice_probe(gpsb200_ctx_t *ctx, const int32_t *prn_in, const double *phase_guess_in, int eager);
int gpsb200_slice_finish(gpsb200_ctx_t *ctx, const int32_t *prn_in, const double *phase_in, int32_t *prn_out,
                         double *phase_out, gpsb200_stats_t *stats);
/* Same with a hand-over callback: invoked with the exact outgoing state as soon as the host scan has it -- for an
 * eager slice BEFORE the long kernels are enqueued, so that a message to the successor (an NCCL send is a kernel too)
 * does not queue behind this slice's own synthesis. */
typedef void (*gpsb200_handoff_fn)(void *user, const int32_t *prn_out, const double *phase_out);
int gpsb200_slice_finish_cb(gpsb200_ctx_t *ctx, const int32_t *prn_in, const double *phase_in, int32_t *prn_out,
                            double *phase_out, gpsb200_stats_t *stats, gpsb200_handoff_fn handoff, void *user);
/* Host only: the link of a slice from its parameters alone (identical to what gpsb200_slice_prepare fills). */
int gpsb200_slice_link_host(const gpsb200_chan_t *chans, int nblk, int nchan, gpsb200_slice_link_t *link);
/* Host only: (prn_in, phase_in) -> guessed (prn_out, phase_out) after the slice `link` describes. */
int gpsb200_link_apply(const gpsb200_slice_link_t *link, int nchan, const int32_t *prn_in, const double *phase_in,
                       int32_t *prn_out, double *phase_out);
/* The same two for either carrier NCO (carrier_nco = GPSB200_CARRIER_FP64 / _U32; the two functions above are the FP64
 * forms). U32: link.value is the EXACT advance over the slice modulo 2^32 (or, with reset_inside, the exact absolute
 * phase after it), so gpsb200_link_apply_nco yields exact, not guessed, outgoing states; phases are u32 accumulators. */
int gpsb200_slice_link_host_nco(const gpsb200_chan_t *chans, int nblk, int nchan, int carrier_nco,
                                gpsb200_slice_link_t *link);
int gpsb200_link_apply_nco(const gpsb200_slice_link_t *link, int nchan, int carrier_nco, const int32_t *prn_in,
                           const double *phase_in, int32_t *prn_out, double *phase_out);

/* Test hook of the device self-check: corrupt the resolved carrier chain of the next calls by one unit of the
 * rounding grid (on != 0); every synth call must then fail with GPSB200_ERR_INTERNAL instead of returning samples.
 * A GPSB200_CARRIER_U32 context has no carrier chain to corrupt: GPSB200_ERR_ARG. */
int gpsb200_debug_corrupt_chain(gpsb200_ctx_t *ctx, int on);

/* Name of the synthesis kernel a call with nchan channels launches on this context as it stands: "k_synth_lanes"
 * (lane = sample: run length a multiple of 96 up to 2400, every code rate seen so far within 1.0157 .. 1.0302 MHz, 16-byte aligned
 * destination, GPSB200_LANES != 0) or "k_synth" (lane = channel, no such conditions); "k_synth_lanes_u32" / "k_synth_u32" in a
 * GPSB200_CARRIER_U32 context (same selection rule). Both are bit-exact; for reporting. */
const char *gpsb200_synth_kernel_name(const gpsb200_ctx_t *ctx, int nchan);

/* Re-run the device part of the previous gpsb200_synth_blocks_device call (parameters,
 * start phases and guesses already resident in HBM): used by bench.py to time the kernels
 * alone. kernel_mask bits: 8 = carrier tables, 4 = carrier probe, 1 = run checkpoints, 2 = synthesis. */
int gpsb200_replay_device(gpsb200_ctx_t *ctx, void *dst_device, void *stream, int kernel_mask);

/* Exact carrier phase after n samples of Doppler f_carr (the chain of gps.c:2821-2826
 * without stepping every sample); host-only helper, also used by time-slice sharding
 * to seed a rank's first block. FP64 carrier NCO only (the U32 one is u + n * step modulo 2^32). */
double gpsb200_carrier_advance(double carr_phase, double f_carr, int64_t nsamples);

/* Exact carrier phases after nblk blocks for every channel slot (same chaining rule as
 * gpsb200_synth_blocks; phase_in == NULL: block 0 takes chans[0][c].carr_phase, else
 * phase_in[c] continues a previous call). Host only, `threads` worker threads. A rank of a
 * time-slice sharded run calls this on the blocks BEFORE its slice to seed its first block.
 * FP64 carrier NCO only (for U32 use gpsb200_slice_link_host_nco + gpsb200_link_apply_nco: exact). */
int gpsb200_carrier_chain(const gpsb200_chan_t *chans, int nblk, int nchan, const double *phase_in,
                          double *phase_out, int threads);

/* Same result as gpsb200_carrier_chain, but resolved with the context's parallel-in-time machinery
 * (device probe kernel + host fix-up scan, no synthesis): ~6 ms per 3000 blocks x 32 channels
 * instead of seconds of sequential host walking. nblk may exceed cfg.max_blocks. A rank of a
 * time-slice sharded run seeds its first block with this. */
int gpsb200_carrier_chain_device(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan,
                                 const double *phase_in, double *phase_out);

/* Host-only view of the parallel-in-time carrier chain (what the device probe kernel plus
 * the host fix-up do per block): walk `nsamples` from the GUESSED phase, then derive the exact
 * end phase of the TRUE start phase from it. Returns 1 and *end_out when the speculation is
 * accepted (then *end_out == gpsb200_carrier_advance(start, ...), bit for bit), 0 when it is
 * rejected (the pipeline then walks that block sequentially). For tests. */
int gpsb200_carrier_probe_fixup(double start, double guess, double f_carr, int64_t nsamples, double *end_out);

/* Host-only model of the two-level (span) resolution of the chain for one satellite over nblk blocks with Doppler
 * f_carr[j]: block probes from guesses derived from start_guess, speculative chaining of the span for both parity
 * variants, ONE fix-up with the true start. Returns 1 and the exact start phase of every block plus the end phase
 * (starts_out[nblk + 1]) when the span-level speculation is accepted, 0 when it is rejected (the pipeline then
 * resolves the span block by block). For tests. */
int gpsb200_span_chain_host(const double *f_carr, int nblk, double start_true, double start_guess, double *starts_out);

/* Host model of the lane = sample synthesis kernel (csrc/synth_lanes.h) for ONE block: the same window / band / repair
 * logic, executed on the CPU, int16 I/Q out. force bits: 1 = repair every sample's index, 2 = exact chip signs for every
 * window, 4 = every repair walks exactly from the run anchor, 8 = carry points of every window by the FP64 second
 * opinion instead of the 32-bit estimate, 16 = GPSB200_CARRIER_U32 (carr_phase / carr_out are u32 accumulators; the
 * carrier index is exact, bits 1 and 4 do not apply). counters[4] = fast samples, repaired samples, exactly
 * rebuilt sign windows, exact walks. For tests (the algorithm against the oracle without a GPU); not a product path. */
int gpsb200_lanes_model_block(const gpsb200_chan_t *chans, int nchan, const uint32_t *nav, int run_samples, int force,
                              int16_t *iq, double *carr_out, int64_t *counters);

/* C/A code of prn (1..32) as 0/1 chips (codegen, gps.c:272-309). */
int gpsb200_codegen(int prn, uint8_t ca[GPSB200_CA_LEN]);

/* ---- scenario engine: the reference's host path outside the sample loop -------------
 * RINEX-2/3 navigation file (plain or gzip-compressed, read through zlib like the reference, gps.c:1147) +
 * location/motion -> the gpsb200_chan_t records and NAV frames the
 * synthesis consumes; bit-identical to what the reference's producer computes (RINEX reader
 * gps.c:1131-1505, satpos/computeRange/ionosphericDelay gps.c:508-611,1893-2026,
 * computeCodePhase gps.c:2033-2064, eph2sbf/generateNavMsg/computeChecksum gps.c:617-884,
 * 1008-1072,2066-2140, allocateChannel gps.c:2142-2235, the 10 Hz / 30 s loop gps.c:2703-2765,
 * 2870-2932). With almanac_file, the almanac pages of subframes 4 and 5 are filled from that SEM file exactly as the
 * reference fills them from its almanac.sem (almanac_read_file almanac.c:73-184, eph2sbf gps.c:772-884); without it,
 * the pages are those of the reference run with its almanac disabled. */
typedef struct gpsb200_scenario_config {
    const char *nav_file;          /* -e: RINEX v2 (or, with rinex3, v3) navigation file */
    const char *motion_file;       /* -m: ECEF motion csv "t,x,y,z" at 10 Hz, NULL = static */
    double lat_deg, lon_deg, height_m;   /* -l */
    int32_t duration_ds;           /* -d in 0.1 s units: (int)(seconds*10+0.5) (gps-sim.c:140); blocks = this - 1 */
    int32_t max_chan;              /* 12 as shipped (gps.h:36); up to 32 */
    int32_t ionosphere_enable;     /* 1 = reference default (-I clears it) */
    int32_t pluto_gain;            /* 1 = gain x 2 (gps.c:2759-2763) */
    int32_t start_year, start_month, start_day, start_hour, start_min;   /* -s; year 0: first ephemeris epoch */
    int32_t rinex3;                /* -3: nav_file is RINEX v3 (gps.c:1512-1891) instead of v2 */
    double start_sec;
    /* -t distance,bearing,height (gps-sim.c:145-148, gps.c:2348-2357): static runs start at a point given by distance
     * [m] and bearing [deg] from the location, height offset [m]; ignored with a motion file, as in the reference */
    int32_t target_valid;
    int32_t carrier_u32;           /* 1: allocation phases of the reference's integer carrier build (gps.c:2212-2213),
                                      carr_phase = (unsigned int) (512.0 * 65536.0 * frac(phase_ini)); 0: FP64 build */
    double target_distance_m, target_bearing_deg, target_height_m;
    /* SEM almanac file (the reference's almanac.sem, gps.c:2614-2651), NULL = no almanac pages (the reference with its
     * almanac disabled). A file that cannot be opened is GPSB200_ERR_ARG; a malformed one is read with the reference's
     * semantics (a parse error before the end of the file drops the whole almanac). A complete record whose toa is more
     * than 4 weeks from the start time is GPSB200_ERR_ARG: the reference writes no block then. Added last in version
     * 0.4: callers must be rebuilt against this header (the struct grew by 8 bytes) */
    const char *almanac_file;
} gpsb200_scenario_config_t;
typedef struct gpsb200_scenario gpsb200_scenario_t;

int gpsb200_scenario_create(const gpsb200_scenario_config_t *cfg, gpsb200_scenario_t **out);
void gpsb200_scenario_destroy(gpsb200_scenario_t *s);
const char *gpsb200_scenario_error(const gpsb200_scenario_t *s);
int gpsb200_scenario_blocks(const gpsb200_scenario_t *s);        /* number of 0.1 s blocks */
int gpsb200_scenario_channels(const gpsb200_scenario_t *s);
int gpsb200_scenario_nav_frames(const gpsb200_scenario_t *s);
const gpsb200_chan_t *gpsb200_scenario_chans(const gpsb200_scenario_t *s);   /* [blocks][channels] */
const uint32_t *gpsb200_scenario_nav(const gpsb200_scenario_t *s);           /* [frames][channels][60] */

/* ---- FIFO / sink boundary: the reference's own API (fifo.h:19-62) --------------
 * Guarded by the reference header's own include guard (fifo.h:13-14), so that a translation unit of the reference
 * that includes both headers -- in either order -- sees the declarations once (they are identical). */
#ifndef FIFO_H
#define FIFO_H
struct iq_buf {
    signed char *data8;        /* 8 bit IQ data  */
    signed short *data16;      /* 16 bit IQ data */
    unsigned int totalLength;  /* allocated size in elements */
    unsigned int validLength;  /* valid elements */
    struct iq_buf *next;
};
bool fifo_create(unsigned buffer_count, unsigned buffer_size, unsigned sample_size);
void fifo_destroy(void);
void fifo_wait_next(void);
void fifo_wait_full(void);
void fifo_halt(void);
struct iq_buf *fifo_acquire(void);
void fifo_enqueue(struct iq_buf *buf);
struct iq_buf *fifo_dequeue(void);
void fifo_release(struct iq_buf *buf);
#endif /* FIFO_H */
/* gpsb200 extension: reproduce the stock reference's loss of buffers 1..6 of a run
 * (tail bug, fifo.c:163-168) so that iqdata.bin is byte-identical to the stock program. The guarantee covers that
 * start-up loss with the reference's geometry (8 buffers, writer started when the FIFO is primed); as in the stock
 * program, further losses while the consumer lags depend on producer/consumer timing. */
void fifo_set_compat_drop(bool on);

/* Feed a contiguous run of I/Q elements into FIFO buffers of whatever size the FIFO was created
 * with, enqueueing each buffer when full and carrying the partly filled one to the next call --
 * the HackRF cadence of the reference (262144-element buffers across 600000-element blocks,
 * gps.c:2847-2856). gpsb200_fifo_push_flush enqueues a remaining partial buffer. */
int gpsb200_fifo_push(const void *elems, size_t count, int sample_size);
int gpsb200_fifo_push_flush(void);

/* iqfile sink (sdr_iqfile.h:16-18 semantics: writes ./iqdata.bin from the FIFO). */
int gpsb200_iqfile_start(const char *path, int sample_size);
void gpsb200_iqfile_stop(void);

#ifdef __cplusplus
}
#endif
#endif /* GPSB200_H */
