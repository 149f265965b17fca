// Device-side data layout and launchers of the GPS L1 C/A synthesis kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gpsb200 {

constexpr int kBlockSamples = 300000;   // sdr.h:26
constexpr int kNavWords = 60;           // gps.h:52
constexpr int kChipWords = 33;          // 1023 chips, periodically extended to 33 x 32 bits
constexpr int kAtabRows = 513;          // carrier table rows; row 512 is never addressed (carr_phase < 1.0 always), a guard

// One record per (block, channel slot), written by the host, read by both kernels.
struct BlockChanDev {
    double c_carr;     // fl(f_carr * delt)  (gps.c:2821)
    double c_code;     // fl(f_code * delt)  (gps.c:2789)
    double gain;       // gps.c:2756
    double carr_in;    // the caller's carr_phase: applies when the slot's satellite differs from the previous block's
    double code0;      // code phase at the first sample (computeCodePhase, gps.c:2049)
    int32_t prn;       // 0 = slot unused
    uint32_t nav0;     // iword | ibit << 8 | icode << 16 at the first sample
    int32_t frame;     // NAV frame index
    // GPSB200_CARRIER_U32 only (zero otherwise): carr_phasestep = (int) round(512.0 * 65536.0 * f_carr * delt)
    // (gps.c:2746) and the exact u32 carrier phase at the block's first sample (host prefix sum, prepare_blocks)
    int32_t step_u32;
    uint32_t u0;
    int32_t pad;
};
static_assert(sizeof(BlockChanDev) == 64, "BlockChanDev layout");

// Exact NCO state at the first sample of a run (run = run_samples consecutive samples).
struct RunCkpt {
    double x;          // carrier phase (U32 contexts: the u32 accumulator as an integer-valued double)
    double y;          // code phase
    uint32_t nav;      // iword | ibit << 8 | icode << 16
    uint32_t pad;
};
static_assert(sizeof(RunCkpt) == 24, "RunCkpt layout");

struct CarrierProbe;          // nco_exact.h
struct SpanBlockState;        // nco_exact.h

// Resolution of one span (span_blocks consecutive blocks) of one channel slot, written by the host scan.
struct SpanRes {
    double start;      // exact carrier phase at the first sample of the span
    double shift;      // regular span: exact start of block j > 0 = speculative start[V] + shift
    int32_t variant;   // V
    int32_t mode;      // 0: regular, 1: per-block exact start phases are in SynthArgs::carr0 (host fallback), 2: idle
};
static_assert(sizeof(SpanRes) == 24, "SpanRes layout");

struct SynthArgs {
    const BlockChanDev *bc;   // [nblk][nchan]
    const double *carr0;      // [nblk][nchan] exact block-start phases of spans the host resolved block by block (mode 1)
    const double *guess;      // [nblk][nchan] guessed start phases for the speculative probe
    CarrierProbe *probe;      // [nblk][nchan] block probes (device copy, read by k_chain)
    CarrierProbe *probe_host; // same, mapped host memory: the host's block-by-block fallback reads them
    CarrierProbe *span_sum;   // [nspan][nchan] span summaries (mapped host memory)
    SpanBlockState *spec;     // [nblk][nchan] speculative block-start phases per variant
    const SpanRes *span_res;  // [nspan][nchan] the host scan's resolution of every span
    int span_blocks, nspan;
    RunCkpt *ck;              // [nblk][nruns][nchan]
    const uint32_t *nav;      // [frames][nav_stride][60]: rows are the context's channel slots (cfg.max_chan >= nchan)
    int nav_stride;
    const uint32_t *chipbits; // [33][33] packed C/A chips per PRN (bit n = ca[n mod 1023]), row 0 unused
    int32_t *atab;            // [nblk][513][32] gain-scaled carrier table per block: I + (Q << 16), column = lane
    double *carr_end;         // [nblk][nchan] carrier phase after the block
    double *last_end_host;    // [nchan], mapped host memory: carrier phase after the LAST block of this launch (self-check
                              // across launches; written by the kernel so that no copy-engine transfer is needed)
    int *chain_errors;        // self-check counter: blocks whose walked end phase != the next block's start phase
    void *out;                // nblk * 600000 int8 or int16
    int nblk, nchan, nruns, run_samples, runs_per_cta, ctas_per_block, iq16;
    int lanes;                // nonzero: calls of at most 16 channels may use k_synth_lanes (every code step in its range)
    int u32;                  // nonzero: GPSB200_CARRIER_U32 context -- the carrier is BlockChanDev::u0 + n * step_u32
                              // modulo 2^32 (RunCkpt::x holds the run start's u32 phase); every kernel of the call
                              // picks its carrier variant from this one flag
};

// Gain-scaled carrier tables of every block (gps.c:2781-2782), fetched by k_synth with TMA bulk copies.
cudaError_t launch_tables(const SynthArgs &a, cudaStream_t s);
// Speculative carrier walk of every (block, channel) from a guessed start phase (nco_exact.h).
cudaError_t launch_probe(const SynthArgs &a, cudaStream_t s);
// Speculative chaining of the block probes inside every span, both parity variants (nco_exact.h: span_chain).
cudaError_t launch_chain(const SynthArgs &a, cudaStream_t s);
// Run-start checkpoints for every (block, channel): exact walk, O(#binade crossings); with a.u32 the code NCO only
// (one thread per (block, channel)), the carrier value of a run start is the closed form.
cudaError_t launch_checkpoints(const SynthArgs &a, cudaStream_t s);
// The per-sample synthesis (gps.c:2767-2857): lanes = channels, warp-sum over channels.
cudaError_t launch_synth(const SynthArgs &a, cudaStream_t s);
// The lane = sample variant for at most 16 channels (synth_lanes.cu); launch_synth() dispatches to it when applicable.
bool synth_lanes_applicable(const SynthArgs &a);
cudaError_t launch_synth_lanes(const SynthArgs &a, cudaStream_t s);
void synth_lanes_launch_shape(const SynthArgs &a, int *ctas, int *threads, size_t *smem);
// Threads per CTA and dynamic shared memory the synthesis launch will use (for reporting).
void synth_launch_shape(const SynthArgs &a, int *ctas, int *threads, size_t *smem);

}  // namespace gpsb200
