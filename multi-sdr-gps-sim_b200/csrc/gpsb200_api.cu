// C ABI of libgpsb200.so (include/gpsb200.h): context, pipeline, host share of the carrier chain.
//
// (k_tables writes the per-block carrier tables k_synth fetches by TMA; it depends on the parameters only.)
// Host work per block and channel is what the reference's 10 Hz path hands to its sample loop
// (gps.c:2731-2765) plus ONE thing the loop carries implicitly: the carrier phase at the start
// of the block, which in the reference is whatever 300000 sequential FP64 additions left behind
// (gps.c:2821-2826). That chain is resolved parallel in time (nco_exact.h): the host GUESSES
// every block's start phase, k_probe walks every block from its guess on the GPU, and a cheap
// sequential host scan (carrier_fixup) turns the probes into exact start phases -- falling back to
// the exact sequential walk for the rare block whose probe cannot be used. Then k_checkpoints and
// k_synth run, in chunks whose download overlaps the synthesis of later chunks.
#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gpsb200.h"
#include "nco_exact.h"
#include "synth_kernels.h"
#include "synth_lanes.h"
#include "synth_tables.h"

using namespace gpsb200;

namespace {

constexpr int kSynthChunk = 256;   // blocks per synthesis launch of the host-destination path (D2H overlap)
constexpr int kSegFirst = 256;     // first carrier-chain segment of the host-destination path: small, so
                                   // that the download can start early ...
constexpr int kSegBlocks = 1024;   // ... later ones larger (their probe kernels are latency bound)
constexpr int kSpanBlocks = 32;    // blocks per span of the two-level carrier chain (nco_exact.h: span_chain)
constexpr int kHostChainBlocks = 2;   // calls of at most this many blocks (the reference's own cadence is ONE block per
                                      // call, gps.c:2703-2865) skip the speculation: the host walks the few NCO chains
                                      // exactly itself (~0.3 ms) instead of two latency-bound kernel round trips

struct ChainState {
    int prn = 0;
    double phase = 0.0;
};

// Small persistent worker pool: the per-segment host passes are sub-millisecond, so thread
// creation per pass would dominate them.
class WorkerPool {
public:
    explicit WorkerPool(int n) {
        for (int i = 0; i < n; i++) th_.emplace_back([this, i] { loop(i); });
    }
    ~WorkerPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    int size() const { return (int) th_.size(); }
    // run job(lo, hi) over [0, n) split into at most size() contiguous ranges; blocks until done
    void run(int n, const std::function<void(int, int)> &job) {
        const int parts = std::max(1, std::min(size(), n));
        if (parts <= 1 || th_.empty()) {
            job(0, n);
            return;
        }
        std::unique_lock<std::mutex> lk(mu_);
        job_ = &job;
        n_ = n;
        parts_ = parts;
        pending_ = parts;
        ++epoch_;
        cv_.notify_all();
        done_.wait(lk, [this] { return pending_ == 0; });
        job_ = nullptr;
    }

private:
    void loop(int id) {
        uint64_t seen = 0;
        for (;;) {
            const std::function<void(int, int)> *job;
            int n, parts;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || epoch_ != seen; });
                if (stop_) return;
                seen = epoch_;
                job = job_;
                n = n_;
                parts = parts_;
            }
            if (id < parts) {
                const int per = (n + parts - 1) / parts, lo = id * per, hi = std::min(n, lo + per);
                if (lo < hi) (*job)(lo, hi);
                std::lock_guard<std::mutex> lk(mu_);
                if (--pending_ == 0) done_.notify_all();
            }
        }
    }
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    const std::function<void(int, int)> *job_ = nullptr;
    int n_ = 0, parts_ = 0, pending_ = 0;
    uint64_t epoch_ = 0;
    bool stop_ = false;
};

}  // namespace

struct gpsb200_ctx {
    gpsb200_config_t cfg{};
    int nruns = 0;
    cudaStream_t s_compute = nullptr, s_copy = nullptr, s_pre = nullptr, s_ck = nullptr;
    // timing events of a call (gpsb200_stats_t): the call's stream, and the first segment's probe and checkpoint kernels
    cudaEvent_t ev_start = nullptr, ev_probe_start = nullptr, ev_probe_end = nullptr, ev_ck_start = nullptr,
                ev_ck_end = nullptr, ev_end = nullptr;
    std::vector<cudaEvent_t> ev_done;      // one per synthesis chunk
    BlockChanDev *d_bc = nullptr, *h_bc = nullptr;
    RunCkpt *d_ck = nullptr, *h_ck = nullptr;          // h_ck: run checkpoints of small calls, computed on the host
    uint32_t *d_nav = nullptr, *h_nav = nullptr;
    uint32_t *d_chips = nullptr;
    int32_t *d_atab = nullptr;             // per-block carrier tables (k_tables -> k_synth)
    double *d_carr_end = nullptr;
    int *d_chain_errors = nullptr, *h_chain_errors = nullptr;   // device self-check of the carrier chain
    double *d_guess = nullptr, *h_guess = nullptr;     // speculative block-start phases
    std::vector<uint8_t> h_guess_abs;                  // relative-mode marker per (block, channel), see prepare_blocks
    std::vector<uint8_t> h_span_flags;                 // per (span, channel): 1 = every block idle, 2 = one satellite throughout
    double *d_carr0 = nullptr, *h_carr0 = nullptr;     // exact block-start phases of host-resolved (irregular) spans
    CarrierProbe *d_probe = nullptr;                   // block probes in HBM (k_chain reads them)
    CarrierProbe *h_probe = nullptr, *d_probe_host = nullptr;   // ... and in mapped host memory (host fallback)
    CarrierProbe *h_span_sum = nullptr, *d_span_sum = nullptr;  // span summaries, mapped host memory
    SpanBlockState *d_spec = nullptr;                  // speculative block-start phases
    bool u32 = false;                                  // cfg.carrier_nco == GPSB200_CARRIER_U32: exact closed-form carrier,
                                                       // none of the carrier-chain stages (probes, chaining, scan) run
    bool lanes_on = true;                              // GPSB200_LANES=0: always k_synth (lane = channel)
    bool lanes_veto = false;                           // a channel record outside k_synth_lanes' range was seen
    SpanRes *d_span_res = nullptr, *h_span_res = nullptr;
    int max_spans = 0, max_segs = 0;
    double *h_seg_end = nullptr, *d_seg_end = nullptr;   // mapped: device-walked end phases of every pipeline segment's last block
    std::vector<double> seg_expect;        // what the chain says they must be
    std::vector<cudaEvent_t> ev_seg;       // probes of segment i complete
    void *const *scatter = nullptr;        // gpsb200_synth_blocks_scatter: one host destination per block
    bool fault_inject_chain = false;
    bool trace_on = false;
    double trace_t0 = 0.0;       // gpsb200_debug_corrupt_chain(): test hook of the device self-check
    // state of a begun, not yet finished call (gpsb200_slice_prepare / gpsb200_slice_finish)
    struct Pending {
        bool active = false;
        int nblk = 0, nchan = 0, sample_size = 0;
        void *dst = nullptr, *dst_host = nullptr;
        cudaStream_t stream = nullptr;
        bool probed = false, finished = false, eager = false;
        int nseg = 0;
        gpsb200_stats_t st{};
    } pending;
    void *d_out = nullptr;
    size_t out_bytes = 0;
    bool nav_dirty = true;
    bool graded_chunks = true;             // GPSB200_GRADED_CHUNKS=0: uniform 256-block chunks (A/B knob)
    std::unique_ptr<WorkerPool> pool;      // host passes (guesses, fix-up scan)
    SynthArgs last{};                      // replay state
    bool have_last = false;
    std::string err;
};

namespace {

std::array<cudaEvent_t *, 6> timing_events(gpsb200_ctx *ctx) {
    return {&ctx->ev_start, &ctx->ev_probe_start, &ctx->ev_probe_end, &ctx->ev_ck_start, &ctx->ev_ck_end, &ctx->ev_end};
}

struct OneSatellite {          // parameter accessor of span_chain() for the host model: one satellite, increments cc[j]
    const double *cc;
    __host__ __device__ void operator()(int j, double &c, int32_t &prn) const {
        c = cc[j];
        prn = 1;
    }
};

double now_ms();
// GPSB200_TRACE=1: host time stamps of the pipeline's phases on stderr (diagnostics)
void trace(gpsb200_ctx *ctx, const char *what);

int fail(gpsb200_ctx *c, int code, const std::string &msg) {
    if (c) c->err = msg;
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(ctx, GPSB200_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

void trace(gpsb200_ctx *ctx, const char *what) {
    if (!ctx->trace_on) return;
    const double t = now_ms();
    fprintf(stderr, "[gpsb200 dev %d +%8.3f ms] %s (%d host workers)\n", ctx->cfg.device, t - ctx->trace_t0, what,
            ctx->pool ? ctx->pool->size() : 0);
}

// Host pre-pass: validate, fill the device-layout records and GUESS every block's start
// carrier phase (closed form + expected rounding drift, long double accumulation).
// Phases as 64-bit fixed point (cycles * 2^64, modulo one cycle) for the closed-form guesses.
inline uint64_t phase_to_fix(double p) { return (p >= 0.0 && p < 1.0) ? (uint64_t) (p * 0x1p64) : 0; }
inline double fix_to_phase(uint64_t a) { return (double) (a >> 11) * 0x1p-53; }
inline uint64_t step_to_fix(double c) {     // c in (-1, 1): c * 2^64 modulo 2^64 (exact for |c| >= 2^-12, else truncated)
    const uint64_t m = (uint64_t) (std::fabs(c) * 0x1p64);
    return c < 0.0 ? (uint64_t) 0 - m : m;
}

inline bool valid_u32_phase(double p) { return p >= 0.0 && p < 4294967296.0 && p == std::floor(p); }

// With link != NULL (time-slice hand-over, gpsb200_slice_prepare) the incoming chain state is not known yet:
// guesses are accumulated RELATIVE to it (h_guess holds the advance since the slice start, h_guess_abs marks
// blocks after a (re)allocation inside the slice, whose guesses are absolute) and finalize_guesses() adds the
// offset later; *link describes how the slice maps an incoming state to the guessed outgoing one.
// end_guess (optional): the GUESSED chain state after block b1-1, to seed the guesses of the next segment when that
// is prepared before this one has been resolved.
// U32 contexts: the same pass computes every block's carr_phasestep and its EXACT start phase (a modular prefix sum that
// restarts from carr_phase whenever the slot's satellite changes); with link != NULL the start phases of blocks before
// the slot's first (re)allocation are relative to the incoming phase (h_guess_abs == 0) until u32_rebase().
int prepare_blocks(gpsb200_ctx *ctx, const gpsb200_chan_t *chans, int b0, int b1, int nchan,
                   const std::vector<ChainState> &chain, gpsb200_slice_link_t *link = nullptr,
                   std::vector<ChainState> *end_guess = nullptr) {
    const double delt = 1.0 / (double) GPSB200_SAMPLERATE;     // gps.c:2298
    const bool u32 = ctx->u32;
    std::vector<int> status(nchan, GPSB200_OK);
    std::vector<uint8_t> lanes_bad(nchan, 0);
    ctx->pool->run(nchan, [&](int c_lo, int c_hi) {
        for (int c = c_lo; c < c_hi; c++) {
            // phase accumulator in cycles * 2^64, modulo 2^64 (= modulo one cycle): exact integer arithmetic
            uint64_t acc = phase_to_fix(chain[c].phase);    // exact phase after block b0-1 (if any)
            uint32_t uacc = u32 ? (uint32_t) chain[c].phase : 0u;   // U32: exact phase after block b0-1
            int prev_prn = chain[c].prn;                    // 0 at the start of a call: block 0 is "fresh"
            bool absolute = link == nullptr;                // relative mode: true once a slot was (re)allocated
            if (link) {
                acc = 0;
                uacc = 0u;
                prev_prn = chans[(size_t) b0 * nchan + c].prn;      // block b0 continues whatever comes in (decided later)
                link->prn_first[c] = prev_prn;
                link->first_phase[c] = prev_prn > 0 ? chans[(size_t) b0 * nchan + c].carr_phase : 0.0;
            }
            int span_first_prn = 0;
            uint8_t span_idle = 1, span_uniform = 1;
            for (int b = b0; b < b1; b++) {
                const gpsb200_chan_t &in = chans[(size_t) b * nchan + c];
                const size_t i = (size_t) b * nchan + c;
                BlockChanDev &o = ctx->h_bc[i];
                memset(&o, 0, sizeof o);
                // what the host scan wants to know about the span this block belongs to (resolve_chain)
                if (b % kSpanBlocks == 0) {
                    span_first_prn = in.prn;
                    span_idle = span_uniform = 1;
                }
                span_idle &= in.prn <= 0;
                span_uniform &= in.prn == span_first_prn;
                if ((b + 1) % kSpanBlocks == 0 || b + 1 == b1)
                    ctx->h_span_flags[(size_t) (b / kSpanBlocks) * nchan + c] = (uint8_t) (span_idle | (span_uniform << 1));
                ctx->h_guess[i] = 0.0;
                ctx->h_guess_abs[i] = absolute ? 1 : 0;
                if (in.prn <= 0) {
                    prev_prn = 0;
                    absolute = true;                        // whatever follows starts from an allocation phase
                    continue;
                }
                if (in.prn > 32 || in.iword < 0 || in.iword >= GPSB200_NAV_WORDS || in.ibit < 0 || in.ibit >= 30 ||
                    in.icode < 0 || in.icode >= 20 || in.nav_frame < 0 || in.nav_frame >= ctx->cfg.max_nav_frames ||
                    !(in.code_phase >= 0.0 && in.code_phase < 1023.0) ||
                    // the per-lane chip window holds 24 chips per 64 samples: f_code <= 1.07 MHz (GPS: 1.023 MHz +- 4 Hz)
                    !(in.f_code > 0.0 && in.f_code <= 1.07e6) ||
                    // one wrap per step keeps the phase in [0,1) only for |f_carr * delt| < 1
                    !(std::isfinite(in.f_carr) && std::fabs(in.f_carr) < 2.9e6) || !std::isfinite(in.gain)) {
                    status[c] = GPSB200_ERR_ARG;
                    return;
                }
                // a slot whose satellite changed (or the first block of a call): the caller's carr_phase applies
                if (!(u32 ? valid_u32_phase(in.carr_phase) : (in.carr_phase >= 0.0 && in.carr_phase < 1.0))) {
                    status[c] = GPSB200_ERR_ARG;      // read whenever a slot takes a new satellite
                    return;
                }
                if (in.prn != prev_prn) {
                    acc = phase_to_fix(in.carr_phase);
                    uacc = u32 ? (uint32_t) in.carr_phase : 0u;
                    absolute = true;
                }
                ctx->h_guess_abs[i] = absolute ? 1 : 0;
                prev_prn = in.prn;
                o.c_carr = in.f_carr * delt;                    // gps.c:2821
                o.c_code = in.f_code * delt;                    // gps.c:2789
                if (!lanes::code_step_ok(o.c_code) || (!u32 && !(std::fabs(o.c_carr) < 0.5))) lanes_bad[c] = 1;
                o.gain = in.gain;
                o.carr_in = in.carr_phase;
                o.code0 = in.code_phase;
                o.prn = in.prn;
                o.nav0 = (uint32_t) in.iword | ((uint32_t) in.ibit << 8) | ((uint32_t) in.icode << 16);
                o.frame = in.nav_frame;
                if (u32) {
                    o.step_u32 = lanes::u32_carrier_step(in.f_carr);
                    o.u0 = uacc;
                    uacc += (uint32_t) GPSB200_BLOCK_SAMPLES * (uint32_t) o.step_u32;     // gps.c:2828, modulo 2^32
                    continue;
                }
                ctx->h_guess[i] = fix_to_phase(acc);
                // one block: 300000 steps of c, plus the expected rounding drift of those steps. (The drift of a block is
                // up to +-8e-12 cycles and depends on the low bits of c, i.e. it is uncorrelated from block to block:
                // evaluating it for every 4th block only was tried and made 50x more probes miss.)
                acc += (uint64_t) GPSB200_BLOCK_SAMPLES * step_to_fix(o.c_carr);
                acc += (uint64_t) (int64_t) ((double) GPSB200_BLOCK_SAMPLES * carrier_drift_per_step(o.c_carr) * 0x1p64);
            }
            const double end_phase = u32 ? (double) uacc : fix_to_phase(acc);
            if (end_guess) {
                (*end_guess)[c].prn = prev_prn > 0 ? prev_prn : 0;
                (*end_guess)[c].phase = prev_prn > 0 ? end_phase : 0.0;
            }
            if (link) {
                link->prn_last[c] = prev_prn > 0 ? prev_prn : 0;
                link->reset_inside[c] = absolute ? 1 : 0;
                link->value[c] = end_phase;
            }
        }
    });
    for (int c = 0; c < nchan; c++)
        if (status[c] != GPSB200_OK) return fail(ctx, status[c], "invalid channel parameters in slot " + std::to_string(c));
    // k_synth_lanes covers every code rate a GPS receiver can see (1.0157 .. 1.0302 MHz); anything else keeps this
    // context on k_synth from here on (both are exact; the choice is sticky so that no launch mixes assumptions)
    for (int c = 0; c < nchan; c++)
        if (lanes_bad[c]) ctx->lanes_veto = true;
    // The reference stores (short)i_acc (gps.c:2834); the packed I/Q accumulation is
    // exact as long as |acc| stays inside int16, which bounds the sum of amplitudes.
    for (int b = b0; b < b1; b++) {
        double amp = 0.0;
        for (int c = 0; c < nchan; c++) amp += std::fabs(ctx->h_bc[(size_t) b * nchan + c].gain) * 250.0;
        if (amp > 32767.0) return fail(ctx, GPSB200_ERR_RANGE, "sum of channel amplitudes exceeds int16 range");
    }
    return GPSB200_OK;
}

// U32: the exact chain state after block b1-1, straight from the prepared records (closed form).
void u32_chain_end(const gpsb200_ctx *ctx, int b1, int nchan, std::vector<ChainState> &chain) {
    for (int c = 0; c < nchan; c++) {
        const BlockChanDev &p = ctx->h_bc[(size_t) (b1 - 1) * nchan + c];
        chain[c].prn = p.prn > 0 ? p.prn : 0;
        chain[c].phase = p.prn > 0 ? (double) (p.u0 + (uint32_t) GPSB200_BLOCK_SAMPLES * (uint32_t) p.step_u32) : 0.0;
    }
}

// U32, relative mode of a slice: the exact incoming state is known now; move the start phases of the blocks before each
// slot's first (re)allocation from "advance since the slice start" to absolute (same rule as finalize_guesses).
void u32_rebase(gpsb200_ctx *ctx, int nblk, int nchan, const int32_t *prn_in, const double *phase_in) {
    for (int c = 0; c < nchan; c++) {
        const BlockChanDev &first = ctx->h_bc[c];
        const bool cont = prn_in && phase_in && first.prn > 0 && prn_in[c] == first.prn;
        const uint32_t off = (uint32_t) (cont ? phase_in[c] : first.carr_in);
        for (int b = 0; b < nblk; b++) {
            const size_t i = (size_t) b * nchan + c;
            if (ctx->h_guess_abs[i] || ctx->h_bc[i].prn <= 0) continue;
            ctx->h_bc[i].u0 += off;
        }
    }
}

// Incoming carrier phases a caller hands in (slots with prn_in > 0): [0,1) for FP64, u32 accumulators for U32.
bool phases_ok(const gpsb200_ctx *ctx, int nchan, const int32_t *prn_in, const double *phase_in) {
    if (!prn_in || !phase_in) return true;
    for (int c = 0; c < nchan; c++)
        if (prn_in[c] > 0 && !(ctx->u32 ? valid_u32_phase(phase_in[c]) : (phase_in[c] >= 0.0 && phase_in[c] < 1.0))) return false;
    return true;
}

// Second pass of the relative mode: the (guessed) incoming state is known now. (U32 contexts guess nothing: their
// start phases are exact and are rebased once the exact incoming state is known, u32_rebase.)
void finalize_guesses(gpsb200_ctx *ctx, int b0, int b1, int nchan, const int32_t *prn_in, const double *phase_in) {
    if (ctx->u32) return;
    ctx->pool->run(nchan, [&](int c_lo, int c_hi) {
        for (int c = c_lo; c < c_hi; c++) {
            const BlockChanDev &first = ctx->h_bc[(size_t) b0 * nchan + c];
            const bool cont = prn_in && phase_in && first.prn > 0 && prn_in[c] == first.prn;
            const double off = cont ? phase_in[c] : first.carr_in;
            for (int b = b0; b < b1; b++) {
                const size_t i = (size_t) b * nchan + c;
                if (ctx->h_guess_abs[i] || ctx->h_bc[i].prn <= 0) continue;
                double g = ctx->h_guess[i] + off;
                if (g >= 1.0) g -= 1.0;
                if (!(g >= 0.0 && g < 1.0)) g = 0.0;
                ctx->h_guess[i] = g;
            }
        }
    });
}

// The exact chain state after block b0-1 is known: move the guesses of blocks [b0, b1) by the error the guess of
// block b0 turned out to have (a slot's guesses are corrected up to its next (re)allocation, whose phase is exact).
void reanchor_guesses(gpsb200_ctx *ctx, int b0, int b1, int nchan, const std::vector<ChainState> &chain) {
    ctx->pool->run(nchan, [&](int c_lo, int c_hi) {
        for (int c = c_lo; c < c_hi; c++) {
            const BlockChanDev &first = ctx->h_bc[(size_t) b0 * nchan + c];
            if (first.prn <= 0 || chain[c].prn != first.prn) continue;     // starts from an allocation phase: exact already
            double delta = chain[c].phase - ctx->h_guess[(size_t) b0 * nchan + c];
            if (delta > 0.5) delta -= 1.0;
            if (delta < -0.5) delta += 1.0;
            for (int b = b0; b < b1; b++) {
                const size_t i = (size_t) b * nchan + c;
                if (ctx->h_bc[i].prn != first.prn) break;
                double g = ctx->h_guess[i] + delta;
                if (g >= 1.0) g -= 1.0;
                if (g < 0.0) g += 1.0;
                if (!(g >= 0.0 && g < 1.0)) g = 0.0;
                ctx->h_guess[i] = g;
            }
        }
    });
}

// One block of the chain, resolved on the host from its block probe (the first level of the speculation);
// the exact sequential walk when the probe cannot be used. Returns 1 when it had to walk.
inline int resolve_block(ChainState &st, const BlockChanDev &bc, const CarrierProbe &probe, double &start_out) {
    if (bc.prn <= 0) {
        st.prn = 0;
        start_out = 0.0;
        return 0;
    }
    if (st.prn != bc.prn) st.phase = bc.carr_in;
    st.prn = bc.prn;
    start_out = st.phase;
    double xe;
    if (carrier_fixup(st.phase, bc.c_carr, probe, xe)) {
        st.phase = xe;
        return 0;
    }
    int64_t dummy = 0;
    nco_advance<NCO_CARRIER>(st.phase, bc.c_carr, GPSB200_BLOCK_SAMPLES, dummy);
    return 1;
}

// Host scan of the two-level chain for blocks [b0, b1) (b0 is a span boundary of this launch): one
// carrier_fixup per SPAN from the span summaries k_chain left in mapped host memory; a span the device
// could not chain speculatively (reallocation inside it, Doppler zero crossing, a rejected block probe)
// or whose summary does not fit the true start phase is resolved block by block from the block probes.
// Serial over spans per channel, parallel over channels. Returns the number of blocks walked sequentially and adds the
// number of spans resolved block by block to spans_slow.
int64_t resolve_chain(gpsb200_ctx *ctx, int b0, int b1, int nchan, std::vector<ChainState> &chain, int64_t &spans_slow) {
    std::vector<int64_t> fallbacks(nchan, 0), slow(nchan, 0);
    const int K = kSpanBlocks;
    const int nspan = (b1 - b0 + K - 1) / K;
    ctx->pool->run(nchan, [&](int c_lo, int c_hi) {
        for (int c = c_lo; c < c_hi; c++) {
            ChainState st = chain[c];
            for (int sp = 0; sp < nspan; sp++) {
                const int s0 = b0 + sp * K, s1 = std::min(b1, s0 + K);
                SpanRes &res = ctx->h_span_res[(size_t) (s0 / K) * nchan + c];
                const BlockChanDev &first = ctx->h_bc[(size_t) s0 * nchan + c];
                const uint8_t flags = ctx->h_span_flags[(size_t) (s0 / K) * nchan + c];     // from prepare_blocks
                const bool idle = flags & 1, uniform = flags & 2;
                res.start = res.shift = 0.0;
                res.variant = 0;
                if (idle) {
                    res.mode = 2;
                    st.prn = 0;
                    continue;
                }
                if (uniform && first.prn > 0) {
                    const double start = st.prn == first.prn ? st.phase : first.carr_in;
                    const CarrierProbe &sum = ctx->h_span_sum[(size_t) (s0 / K) * nchan + c];
                    double xe, d;
                    int v;
                    if (carrier_fixup(start, first.c_carr, sum, xe, &v, &d, 1.0)) {
                        res.mode = 0;
                        res.start = start;
                        res.shift = d;
                        res.variant = v;
                        st.prn = first.prn;
                        st.phase = xe;
                        continue;
                    }
                }
                // block by block (first level only)
                res.mode = 1;
                ++slow[c];
                for (int b = s0; b < s1; b++) {
                    const size_t i = (size_t) b * nchan + c;
                    fallbacks[c] += resolve_block(st, ctx->h_bc[i], ctx->h_probe[i], ctx->h_carr0[i]);
                }
            }
            chain[c] = st;
        }
    });
    // test hook of the device self-check (gpsb200_debug_corrupt_chain): corrupt the resolution of one span by
    // one unit of the rounding grid; k_checkpoints must notice
    if (ctx->fault_inject_chain && b1 - b0 > 6) {
        SpanRes &r = ctx->h_span_res[(size_t) (b0 / K) * nchan];
        if (r.mode == 0) r.shift += 0x1p-51;
        else if (r.mode == 1) ctx->h_carr0[(size_t) (b0 + 5) * nchan] += 0x1p-51;
    }
    int64_t n = 0;
    for (int c = 0; c < nchan; c++) {
        n += fallbacks[c];
        spans_slow += slow[c];
    }
    return n;
}

// Kernel arguments for blocks [blk0, blk1) of a call whose samples go to dst (block 0 of the call; kernels that write no
// samples need neither dst nor the sample size).
SynthArgs args_of(gpsb200_ctx *ctx, int blk0, int blk1, int nchan, int sample_size = GPSB200_SC08, void *dst = nullptr) {
    // blk0 is a multiple of kSpanBlocks whenever the chain kernels are launched with these arguments
    const int nblk = blk1 - blk0;
    const size_t off = (size_t) blk0 * nchan;
    SynthArgs a{};
    a.bc = ctx->d_bc + off;
    a.carr0 = ctx->d_carr0 + off;
    a.guess = ctx->d_guess + off;
    a.probe = ctx->d_probe + off;
    a.probe_host = ctx->d_probe_host + off;
    a.spec = ctx->d_spec + off;
    a.span_blocks = kSpanBlocks;
    a.nspan = (nblk + kSpanBlocks - 1) / kSpanBlocks;
    a.span_sum = ctx->d_span_sum + (size_t) (blk0 / kSpanBlocks) * nchan;
    a.span_res = ctx->d_span_res + (size_t) (blk0 / kSpanBlocks) * nchan;
    a.ck = ctx->d_ck + off * ctx->nruns;
    a.nav = ctx->d_nav;
    a.nav_stride = ctx->cfg.max_chan;
    a.chipbits = ctx->d_chips;
    a.atab = ctx->d_atab + (size_t) blk0 * kAtabRows * 32;
    a.carr_end = ctx->d_carr_end + off;
    a.chain_errors = ctx->d_chain_errors;
    a.out = dst ? (char *) dst + (size_t) blk0 * GPSB200_BLOCK_ELEMS * sample_size : nullptr;
    a.nblk = nblk;
    a.nchan = nchan;
    a.nruns = ctx->nruns;
    a.run_samples = ctx->cfg.run_samples;
    a.iq16 = sample_size == GPSB200_SC16;
    a.lanes = ctx->lanes_on && !ctx->lanes_veto ? 1 : 0;
    a.u32 = ctx->u32 ? 1 : 0;
    // lanes per run follow the channel count; a CTA takes up to 24 warps' worth of runs
    const int grp = nchan > 16 ? 32 : (nchan > 8 ? 16 : 8);
    const int rpw = 32 / grp;
    int per_cta = 24 * rpw;
    const int ctas = (ctx->nruns + per_cta - 1) / per_cta;
    per_cta = (ctx->nruns + ctas - 1) / ctas;
    a.runs_per_cta = per_cta;
    a.ctas_per_block = ctas;
    return a;
}

int upload_nav(gpsb200_ctx *ctx, cudaStream_t s) {
    if (!ctx->nav_dirty) return GPSB200_OK;
    const size_t bytes = (size_t) ctx->cfg.max_nav_frames * ctx->cfg.max_chan * GPSB200_NAV_WORDS * 4;
    CU(cudaMemcpyAsync(ctx->d_nav, ctx->h_nav, bytes, cudaMemcpyHostToDevice, s));
    ctx->nav_dirty = false;
    return GPSB200_OK;
}

int check_call(gpsb200_ctx *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size, void *dst) {
    if (!ctx) return GPSB200_ERR_ARG;
    if (!chans || !dst || nblk < 1 || nblk > ctx->cfg.max_blocks || nchan < 1 || nchan > ctx->cfg.max_chan ||
        (sample_size != GPSB200_SC08 && sample_size != GPSB200_SC16))
        return fail(ctx, GPSB200_ERR_ARG, "bad arguments (1 <= nchan <= cfg.max_chan; 1 <= nblk <= cfg.max_blocks)");
    if (!ctx->s_compute) return fail(ctx, GPSB200_ERR_CUDA, "context has no CUDA device");
    if (ctx->pending.active) return fail(ctx, GPSB200_ERR_ARG, "a call begun with gpsb200_slice_prepare has not been finished");
    CU(cudaSetDevice(ctx->cfg.device));     // the caller may be a thread that never selected the context's device
    return GPSB200_OK;
}

// Wait for everything this context has in flight once a call failed with rc (the caller may free its buffers once it
// sees the error code, so no copy into them may still be pending); the error text stays that of rc.
int drained(gpsb200_ctx *ctx, int rc, cudaStream_t extra) {
    if (rc == GPSB200_OK) return rc;
    if (extra) cudaStreamSynchronize(extra);
    cudaStreamSynchronize(ctx->s_compute);
    cudaStreamSynchronize(ctx->s_pre);
    if (ctx->s_ck) cudaStreamSynchronize(ctx->s_ck);
    cudaStreamSynchronize(ctx->s_copy);
    return rc;
}

// The context's own device buffer that results for a host destination are staged in: room for cfg.max_blocks blocks.
int stage_out(gpsb200_ctx *ctx, int sample_size) {
    const size_t need = (size_t) ctx->cfg.max_blocks * GPSB200_BLOCK_ELEMS * sample_size;
    if (ctx->out_bytes >= need) return GPSB200_OK;
    cudaFree(ctx->d_out);
    ctx->d_out = nullptr;
    ctx->out_bytes = 0;
    CU(cudaMalloc(&ctx->d_out, need));
    ctx->out_bytes = need;
    return GPSB200_OK;
}

// The steps of a pipeline segment [b0, b1), which every driver strings together:
//   segment_params -> speculate -> scan -> checkpoints -> synthesize.

// Host records + guesses, parameters up, carrier tables.
int segment_params(gpsb200_ctx *ctx, const gpsb200_chan_t *chans, int b0, int b1, int nchan, cudaStream_t sp,
                   const std::vector<ChainState> &chain, gpsb200_stats_t &st, gpsb200_slice_link_t *link = nullptr,
                   std::vector<ChainState> *end_guess = nullptr) {
    const size_t off = (size_t) b0 * nchan, cnt = (size_t) (b1 - b0) * nchan;
    double t0 = now_ms();
    int rc = prepare_blocks(ctx, chans, b0, b1, nchan, chain, link, end_guess);
    if (rc) return rc;
    st.host_chain_ms += now_ms() - t0;
    CU(cudaMemcpyAsync(ctx->d_bc + off, ctx->h_bc + off, cnt * sizeof(BlockChanDev), cudaMemcpyHostToDevice, sp));
    CU(launch_tables(args_of(ctx, b0, b1, nchan), sp));     // needs only the parameters: off the chain's critical path
    st.launches += 1;
    st.h2d_bytes += (int64_t) (cnt * sizeof(BlockChanDev));
    return GPSB200_OK;
}

// Everything speculative, on stream sp: guesses up, block probes, span chaining, then `probed` is recorded. Needs no
// true start phase. A U32 context has nothing to speculate about (exact closed form).
int speculate(gpsb200_ctx *ctx, int b0, int b1, int nchan, cudaStream_t sp, gpsb200_stats_t &st, bool first,
              cudaEvent_t probed) {
    if (ctx->u32) return GPSB200_OK;
    const size_t off = (size_t) b0 * nchan, cnt = (size_t) (b1 - b0) * nchan;
    const SynthArgs a = args_of(ctx, b0, b1, nchan);
    CU(cudaMemcpyAsync(ctx->d_guess + off, ctx->h_guess + off, cnt * sizeof(double), cudaMemcpyHostToDevice, sp));
    if (first) CU(cudaEventRecord(ctx->ev_probe_start, sp));
    CU(launch_probe(a, sp));
    CU(launch_chain(a, sp));
    if (first) CU(cudaEventRecord(ctx->ev_probe_end, sp));
    CU(cudaEventRecord(probed, sp));
    st.launches += 2;
    st.h2d_bytes += (int64_t) (cnt * sizeof(double));
    st.d2h_bytes += (int64_t) (cnt * sizeof(CarrierProbe) + (size_t) a.nspan * nchan * sizeof(CarrierProbe));
    return GPSB200_OK;
}

// Host scan: chain goes from the exact state after block b0-1 to the one after block b1-1, from the probes and span
// summaries in mapped host memory once `probed` is complete; slow = spans resolved block by block. A U32 context reads
// the exact state off the prepared records (closed form): there are no probes to wait for.
int scan(gpsb200_ctx *ctx, int b0, int b1, int nchan, std::vector<ChainState> &chain, gpsb200_stats_t &st,
         cudaEvent_t probed, int64_t &slow) {
    slow = 0;
    if (ctx->u32) {
        u32_chain_end(ctx, b1, nchan, chain);
        return GPSB200_OK;
    }
    CU(cudaEventSynchronize(probed));
    const double t0 = now_ms();
    st.chain_fallbacks += (int32_t) resolve_chain(ctx, b0, b1, nchan, chain, slow);
    st.host_chain_ms += now_ms() - t0;
    return GPSB200_OK;
}

// Device part of the resolution, on stream sp: the scan's resolutions up, exact run checkpoints (+ the per-block
// self-check). The launch also stores the walked end phases of the segment's last block into row iseg of h_seg_end
// (mapped memory: a copy-engine transfer would queue behind the large result downloads); chain_after, the scan's state
// after block b1-1, is what they must be. verify_chain() compares the two: the self-check across segment and call
// boundaries. After this step the segment's synthesis may be enqueued behind sp.
int checkpoints(gpsb200_ctx *ctx, int b0, int b1, int nchan, cudaStream_t sp, gpsb200_stats_t &st, bool first,
                int64_t slow, int iseg, const std::vector<ChainState> &chain_after) {
    const size_t off = (size_t) b0 * nchan, cnt = (size_t) (b1 - b0) * nchan;
    SynthArgs a = args_of(ctx, b0, b1, nchan);
    const size_t soff = (size_t) (b0 / kSpanBlocks) * nchan, scnt = (size_t) a.nspan * nchan;
    if (first) CU(cudaEventRecord(ctx->ev_ck_start, sp));
    if (!ctx->u32) {                                 // U32: k_checkpoints reads no span resolutions
        CU(cudaMemcpyAsync(ctx->d_span_res + soff, ctx->h_span_res + soff, scnt * sizeof(SpanRes), cudaMemcpyHostToDevice, sp));
        st.h2d_bytes += (int64_t) (scnt * sizeof(SpanRes));
    }
    if (slow > 0) {                                  // rare: per-block start phases of the host-resolved spans
        CU(cudaMemcpyAsync(ctx->d_carr0 + off, ctx->h_carr0 + off, cnt * sizeof(double), cudaMemcpyHostToDevice, sp));
        st.h2d_bytes += (int64_t) (cnt * sizeof(double));
    }
    const bool noted = iseg < ctx->max_segs;
    a.last_end_host = noted ? ctx->d_seg_end + (size_t) iseg * nchan : nullptr;
    CU(launch_checkpoints(a, sp));
    if (first) CU(cudaEventRecord(ctx->ev_ck_end, sp));
    st.launches += 1;
    for (int c = 0; noted && c < nchan; c++) {
        const bool live = chain_after[c].prn > 0 && ctx->h_bc[(size_t) (b1 - 1) * nchan + c].prn == chain_after[c].prn;
        ctx->seg_expect[(size_t) iseg * nchan + c] = live ? chain_after[c].phase : -1.0;       // -1: nothing to compare
    }
    return GPSB200_OK;
}

// Blocks [b0, b0 + nb) from src (the device copy of block b0) to the host on stream s: into the contiguous buffer
// dst_host or, when ctx->scatter is set, every block into its own destination.
int download(gpsb200_ctx *ctx, const char *src, int b0, int nb, int sample_size, void *dst_host, cudaStream_t s,
             gpsb200_stats_t &st) {
    const size_t blk_bytes = (size_t) GPSB200_BLOCK_ELEMS * sample_size;
    if (ctx->scatter) {          // every block straight into its own (FIFO) buffer
        for (int b = b0; b < b0 + nb; b++)
            CU(cudaMemcpyAsync(ctx->scatter[b], src + (size_t) (b - b0) * blk_bytes, blk_bytes, cudaMemcpyDeviceToHost, s));
    } else {
        CU(cudaMemcpyAsync((char *) dst_host + (size_t) b0 * blk_bytes, src, (size_t) nb * blk_bytes, cudaMemcpyDeviceToHost,
                           s));
    }
    st.d2h_bytes += (int64_t) nb * (int64_t) blk_bytes;
    return GPSB200_OK;
}

// Synthesis of blocks [b0, b1) in chunks, each chunk's download to dst_host enqueued on s_copy behind it.
int synth_chunks(gpsb200_ctx *ctx, int b0, int b1, int nchan, int sample_size, void *dst_dev, void *dst_host,
                 cudaStream_t s, gpsb200_stats_t &st, int &ichunk) {
    // the very first chunks are short, so that the download (the long pole of this path) starts early
    for (int c0 = b0, nc = 0; c0 < b1; c0 += nc, ichunk++) {
        nc = kSynthChunk;
        if (ctx->graded_chunks) nc = c0 == 0 ? 32 : (c0 == 32 ? 96 : (c0 == 128 ? 128 : kSynthChunk));
        nc = std::min(nc, b1 - c0);
        const SynthArgs ac = args_of(ctx, c0, c0 + nc, nchan, sample_size, dst_dev);
        CU(launch_synth(ac, s));
        st.launches += 1;
        CU(cudaEventRecord(ctx->ev_done[ichunk], s));
        CU(cudaStreamWaitEvent(ctx->s_copy, ctx->ev_done[ichunk], 0));
        const int rc = download(ctx, (const char *) ac.out, c0, nc, sample_size, dst_host, ctx->s_copy, st);
        if (rc) return rc;
    }
    return GPSB200_OK;
}

// Synthesis of the segment on stream s, behind the checkpoints enqueued on sk; with a host destination in chunks whose
// downloads overlap the synthesis of later chunks.
int synthesize(gpsb200_ctx *ctx, int b0, int b1, int nchan, int sample_size, void *dst_dev, void *dst_host,
               cudaStream_t sk, cudaStream_t s, gpsb200_stats_t &st, int &ichunk) {
    CU(cudaEventRecord(ctx->ev_done[ichunk], sk));
    CU(cudaStreamWaitEvent(s, ctx->ev_done[ichunk], 0));
    ichunk++;
    if (dst_host) return synth_chunks(ctx, b0, b1, nchan, sample_size, dst_dev, dst_host, s, st, ichunk);
    CU(launch_synth(args_of(ctx, b0, b1, nchan, sample_size, dst_dev), s));
    st.launches += 1;
    return GPSB200_OK;
}

void seed_chain(std::vector<ChainState> &chain, int nchan, const int32_t *prn_in, const double *phase_in) {
    for (int c = 0; c < nchan; c++) {
        chain[c].prn = (prn_in && phase_in && prn_in[c] > 0) ? prn_in[c] : 0;
        chain[c].phase = chain[c].prn ? phase_in[c] : 0.0;
    }
}

void export_chain(const std::vector<ChainState> &chain, int nchan, int32_t *prn_out, double *phase_out) {
    for (int c = 0; c < nchan; c++) {
        if (prn_out) prn_out[c] = chain[c].prn;
        if (phase_out) phase_out[c] = chain[c].prn > 0 ? chain[c].phase : 0.0;
    }
}

// A call of one or two blocks (the reference's cadence): the host walks every NCO chain exactly (nco_exact.h) and
// hands the device ready-made run checkpoints; tables + synthesis are the only kernels. Exact by construction.
int small_call(gpsb200_ctx *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size, void *dst_dev,
               void *dst_host, cudaStream_t s, std::vector<ChainState> &chain, int32_t *prn_out, double *carr_phase_out,
               gpsb200_stats_t *stats) {
    gpsb200_stats_t st{};
    double t0 = now_ms();
    int rc = prepare_blocks(ctx, chans, 0, nblk, nchan, chain);
    if (rc) return rc;
    const int nruns = ctx->nruns, run = ctx->cfg.run_samples;
    ctx->pool->run(nchan, [&](int c_lo, int c_hi) {
        for (int c = c_lo; c < c_hi; c++) {
            ChainState stc = chain[c];
            for (int b = 0; b < nblk; b++) {
                const BlockChanDev &p = ctx->h_bc[(size_t) b * nchan + c];
                RunCkpt *ck = ctx->h_ck + (size_t) b * nruns * nchan + c;
                if (p.prn <= 0) {
                    stc.prn = 0;
                    for (int r = 0; r < nruns; r++) ck[(size_t) r * nchan] = RunCkpt{0.0, 0.0, 0u, 0u};
                    continue;
                }
                if (stc.prn != p.prn) stc.phase = p.carr_in;
                stc.prn = p.prn;
                double x = ctx->u32 ? (double) p.u0 : stc.phase, y = p.code0;
                int iword = p.nav0 & 0xFF, ibit = (p.nav0 >> 8) & 0xFF, icode = (p.nav0 >> 16) & 0xFF;
                for (int r = 0; r < nruns; r++) {
                    ck[(size_t) r * nchan] = RunCkpt{x, y, (uint32_t) iword | ((uint32_t) ibit << 8) | ((uint32_t) icode << 16), 0u};
                    int64_t periods = 0, dummy = 0;
                    if (ctx->u32) x = (double) ((uint32_t) x + (uint32_t) run * (uint32_t) p.step_u32);     // gps.c:2828
                    else nco_advance<NCO_CARRIER>(x, p.c_carr, run, dummy);
                    nco_advance<NCO_CODE>(y, p.c_code, run, periods);
                    nav_advance(iword, ibit, icode, periods);
                }
                stc.phase = x;
            }
            chain[c] = stc;
        }
    });
    st.host_chain_ms = now_ms() - t0;
    rc = upload_nav(ctx, s);
    if (rc) return rc;
    const size_t cnt = (size_t) nblk * nchan;
    CU(cudaEventRecord(ctx->ev_start, s));
    CU(cudaMemcpyAsync(ctx->d_bc, ctx->h_bc, cnt * sizeof(BlockChanDev), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(ctx->d_ck, ctx->h_ck, cnt * nruns * sizeof(RunCkpt), cudaMemcpyHostToDevice, s));
    const SynthArgs a = args_of(ctx, 0, nblk, nchan, sample_size, dst_dev);
    CU(launch_tables(a, s));
    CU(launch_synth(a, s));
    CU(cudaEventRecord(ctx->ev_end, s));
    st.launches = 2;
    st.h2d_bytes = (int64_t) (cnt * (sizeof(BlockChanDev) + nruns * sizeof(RunCkpt)));
    if (dst_host) {
        rc = download(ctx, (const char *) dst_dev, 0, nblk, sample_size, dst_host, s, st);
        if (rc) return rc;
        CU(cudaStreamSynchronize(s));
    }
    ctx->last = a;
    ctx->have_last = false;              // nothing to replay: there were no walk kernels
    export_chain(chain, nchan, prn_out, carr_phase_out);
    if (stats) *stats = st;
    return GPSB200_OK;
}

// Pipeline segments of a call: a short first one (its chain resolution is the lead-in of everything), then long ones.
std::vector<std::pair<int, int>> segments_of(int nblk) {
    std::vector<std::pair<int, int>> v;
    int len = kSegFirst;
    for (int b0 = 0; b0 < nblk; len = kSegBlocks) {
        const int b1 = std::min(nblk, b0 + len);
        v.emplace_back(b0, b1);
        b0 = b1;
    }
    return v;
}

// Verdict of the device self-check (all of sp's work must be complete): the per-block comparisons inside the
// checkpoint launches plus the segment-boundary comparisons.
int verify_chain(gpsb200_ctx *ctx, int nseg, int nchan) {
    int bad = *ctx->h_chain_errors;
    for (int i = 0; i < std::min(nseg, ctx->max_segs); i++)
        for (int c = 0; c < nchan; c++) {
            const double want = ctx->seg_expect[(size_t) i * nchan + c];
            if (want >= 0.0 && f64_bits(want) != f64_bits(ctx->h_seg_end[(size_t) i * nchan + c])) ++bad;
        }
    if (bad != 0)
        return fail(ctx, GPSB200_ERR_INTERNAL, "carrier chain self-check failed on " + std::to_string(bad) + " blocks");
    return GPSB200_OK;
}

// The whole path for nblk blocks, as a pipeline of segments: the carrier-chain resolution of a segment (parameters
// up -> block probes -> span chaining -> host scan over the span summaries -> resolutions up -> run checkpoints)
// runs on the context's high-priority pre-phase stream and therefore CONCURRENTLY with the synthesis kernels of
// earlier segments on the caller's stream (the walk kernels are latency bound and fit beside k_synth's CTAs) and,
// with a host destination, with the downloads of finished chunks. Only the first (short) segment's resolution is
// a lead-in. dst_host == NULL: results stay at dst_dev and the call returns once everything is enqueued and the
// chain self-check has been read.
int run_pipeline_inner(gpsb200_ctx *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size,
                       void *dst_dev, void *dst_host, cudaStream_t s, const int32_t *prn_in, const double *phase_in,
                       int32_t *prn_out, double *carr_phase_out, gpsb200_stats_t *stats) {
    gpsb200_stats_t st{};
    std::vector<ChainState> chain(nchan);
    seed_chain(chain, nchan, prn_in, phase_in);
    ctx->trace_t0 = now_ms();
    trace(ctx, "call");
    if (nblk <= kHostChainBlocks && !ctx->fault_inject_chain)
        return small_call(ctx, chans, nblk, nchan, sample_size, dst_dev, dst_host, s, chain, prn_out, carr_phase_out, stats);
    cudaStream_t sp = ctx->s_pre;                       // stream of the pre-phase
    CU(cudaEventRecord(ctx->ev_start, s));
    CU(cudaStreamWaitEvent(sp, ctx->ev_start, 0));      // earlier work on s may still read the buffers rewritten now
    int rc = upload_nav(ctx, sp);
    if (rc) return rc;
    CU(cudaMemsetAsync(ctx->d_chain_errors, 0, sizeof(int), sp));
    const auto segs = segments_of(nblk);
    const int nseg = (int) segs.size();
    int ichunk = 0, nverify = nseg;
    int64_t slow = 0;
    if (!dst_host) {
        // Device destination: nothing has to leave early, so everything speculative goes first -- the host prepares
        // segment after segment (guesses continue from the GUESSED end of the previous segment) while the GPU already
        // probes the earlier ones -- then the host scans the span summaries, and run checkpoints and synthesis are
        // ONE launch each over the whole call.
        std::vector<ChainState> guess = chain, next(nchan);
        CU(cudaStreamWaitEvent(ctx->s_ck, ctx->ev_start, 0));
        for (int i = 0; i < nseg; i++) {
            // the segments' walk kernels alternate between two streams: their long tails (walk lengths differ by
            // an order of magnitude between satellites) overlap instead of adding up
            cudaStream_t sw = (i & 1) ? ctx->s_ck : sp;
            rc = segment_params(ctx, chans, segs[i].first, segs[i].second, nchan, sw, guess, st, nullptr, &next);
            if (!rc) rc = speculate(ctx, segs[i].first, segs[i].second, nchan, sw, st, i == 0, ctx->ev_seg[i]);
            if (rc) return rc;
            guess = next;
        }
        trace(ctx, "speculative work enqueued");
        for (int i = 0; i < nseg; i++) {
            int64_t sl = 0;
            rc = scan(ctx, segs[i].first, segs[i].second, nchan, chain, st, ctx->ev_seg[i], sl);
            if (rc) return rc;
            slow += sl;
        }
        CU(cudaStreamSynchronize(ctx->s_ck));           // (its last segment's event has been waited for; this orders the
        trace(ctx, "host scan done");                   //  checkpoint launch on sp behind everything on s_ck)
        rc = checkpoints(ctx, 0, nblk, nchan, sp, st, true, slow, 0, chain);
        if (!rc) rc = synthesize(ctx, 0, nblk, nchan, sample_size, dst_dev, nullptr, sp, s, st, ichunk);
        if (rc) return rc;
        nverify = 1;
        trace(ctx, "checkpoints + synthesis enqueued");
    } else {
        for (int i = 0; i < nseg; i++) {
            const int b0 = segs[i].first, b1 = segs[i].second;
            rc = segment_params(ctx, chans, b0, b1, nchan, sp, chain, st);
            if (!rc) rc = speculate(ctx, b0, b1, nchan, sp, st, i == 0, ctx->ev_seg[i]);
            if (!rc) rc = scan(ctx, b0, b1, nchan, chain, st, ctx->ev_seg[i], slow);
            if (!rc) rc = checkpoints(ctx, b0, b1, nchan, sp, st, i == 0, slow, i, chain);
            if (!rc) rc = synthesize(ctx, b0, b1, nchan, sample_size, dst_dev, dst_host, sp, s, st, ichunk);
            if (rc) return rc;
        }
    }
    CU(cudaEventRecord(ctx->ev_end, s));
    ctx->last = args_of(ctx, 0, nblk, nchan, sample_size, dst_dev);
    ctx->have_last = true;
    export_chain(chain, nchan, prn_out, carr_phase_out);
    // the device self-check of the carrier chain is never skipped: a wrong start phase must not produce samples silently
    CU(cudaMemcpyAsync(ctx->h_chain_errors, ctx->d_chain_errors, sizeof(int), cudaMemcpyDeviceToHost, sp));
    CU(cudaStreamSynchronize(sp));
    trace(ctx, "pre-phase stream drained (self-check read)");
    rc = verify_chain(ctx, nverify, nchan);
    if (rc) return rc;
    if (dst_host) {
        CU(cudaStreamSynchronize(s));
        CU(cudaStreamSynchronize(ctx->s_copy));
    }
    if (stats) {
        float ms = 0;
        // per-kernel times of the FIRST segment ...
        if (!ctx->u32) {    // (a U32 call records no probe events)
            cudaEventElapsedTime(&ms, ctx->ev_probe_start, ctx->ev_probe_end);
            st.probe_kernel_ms = ms;
        }
        cudaEventElapsedTime(&ms, ctx->ev_ck_start, ctx->ev_ck_end);
        st.checkpoint_kernel_ms = ms;
        if (dst_host) {      // ... and the whole span of the call's stream (a device-destination call is still running)
            cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_end);
            st.kernel_ms = ms;
        }
        *stats = st;
    }
    return GPSB200_OK;
}

int run_pipeline(gpsb200_ctx *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size,
                 void *dst_dev, void *dst_host, cudaStream_t s, const int32_t *prn_in, const double *phase_in,
                 int32_t *prn_out, double *carr_phase_out, gpsb200_stats_t *stats) {
    // nothing of this call may still be in flight when the caller sees an error
    return drained(ctx,
                   run_pipeline_inner(ctx, chans, nblk, nchan, sample_size, dst_dev, dst_host, s, prn_in, phase_in,
                                      prn_out, carr_phase_out, stats),
                   s);
}

}  // namespace

extern "C" {

const char *gpsb200_version(void) { return "gpsb200 0.4 (sm_100a)"; }

int gpsb200_bind_numa(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, (int) sizeof bus, device) != cudaSuccess) {
        cudaGetLastError();
        return GPSB200_ERR_CUDA;
    }
    for (char *p = bus; *p; ++p) *p = (char) tolower((unsigned char) *p);
    int node = -1;
    if (FILE *f = fopen((std::string("/sys/bus/pci/devices/") + bus + "/numa_node").c_str(), "r")) {
        if (fscanf(f, "%d", &node) != 1) node = -1;
        fclose(f);
    }
    if (node < 0) return -1;
    char list[4096] = {0};
    FILE *f = fopen(("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist").c_str(), "r");
    if (!f) return -1;
    const bool got = fgets(list, sizeof list, f) != nullptr;
    fclose(f);
    if (!got) return -1;
    cpu_set_t cur, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof cur, &cur) != 0) return -1;
    int picked = 0;
    for (const char *p = list; *p && *p != '\n';) {            // "0-31,64-95"
        char *end = nullptr;
        long a = strtol(p, &end, 10), b = a;
        if (end == p) break;
        if (*end == '-') b = strtol(end + 1, &end, 10);
        for (long c = a; c <= b && c < CPU_SETSIZE; c++)
            if (CPU_ISSET((int) c, &cur)) {
                CPU_SET((int) c, &want);
                ++picked;
            }
        p = *end == ',' ? end + 1 : end;
    }
    if (picked == 0 || sched_setaffinity(0, sizeof want, &want) != 0) return -1;
    return node;
}

const char *gpsb200_last_error(const gpsb200_ctx_t *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int gpsb200_codegen(int prn, uint8_t ca[GPSB200_CA_LEN]) { return ca_code(prn, ca) == 0 ? GPSB200_OK : GPSB200_ERR_ARG; }

double gpsb200_carrier_advance(double carr_phase, double f_carr, int64_t nsamples) {
    const double c = f_carr * (1.0 / (double) GPSB200_SAMPLERATE);
    int64_t dummy = 0;
    nco_advance<NCO_CARRIER>(carr_phase, c, nsamples, dummy);
    return carr_phase;
}

int gpsb200_carrier_probe_fixup(double start, double guess, double f_carr, int64_t nsamples, double *end_out) {
    const double c = f_carr * (1.0 / (double) GPSB200_SAMPLERATE);
    CarrierProbe p;
    carrier_probe(guess, c, nsamples, p);
    double xe = 0.0;
    const bool ok = carrier_fixup(start, c, p, xe);
    if (ok && end_out) *end_out = xe;
    return ok ? 1 : 0;
}

int gpsb200_span_chain_host(const double *f_carr, int nblk, double start_true, double start_guess, double *starts_out) {
    // Host-only model of the two-level chain for ONE span of one satellite (what k_probe + k_chain + the host scan
    // do): block probes from closed-form guesses, span_chain() for both variants, one carrier_fixup on the summary.
    if (!f_carr || nblk < 1 || !starts_out) return GPSB200_ERR_ARG;
    const double delt = 1.0 / (double) GPSB200_SAMPLERATE;
    std::vector<CarrierProbe> probes(nblk);
    std::vector<double> cc(nblk);
    std::vector<SpanBlockState> spec(nblk);
    long double acc = start_guess;
    for (int j = 0; j < nblk; j++) {
        cc[j] = f_carr[j] * delt;
        double g = (double) acc;
        if (!(g >= 0.0 && g < 1.0)) g = 0.0;
        carrier_probe(g, cc[j], GPSB200_BLOCK_SAMPLES, probes[j]);
        acc += (long double) GPSB200_BLOCK_SAMPLES * ((long double) cc[j] + (long double) carrier_drift_per_step(cc[j]));
        acc -= floorl(acc);
    }
    CarrierProbe sum{}, part{};
    bool ok[2];
    for (int V = 0; V < 2; V++) {
        span_chain(probes.data(), OneSatellite{cc.data()}, nblk, 1, start_guess, V, part, ok[V], spec.data());
        if (V == 0) {
            sum.x_w = part.x_w;
            sum.n_w = part.n_w;
        }
        sum.x_end[V] = part.x_end[V];
        sum.m_pos[V] = ok[V] ? part.m_pos[V] : 0.0;
        sum.m_neg[V] = ok[V] ? part.m_neg[V] : 0.0;
    }
    double xe, d;
    int v;
    if (!carrier_fixup(start_true, cc[0], sum, xe, &v, &d, 1.0)) return 0;
    starts_out[0] = start_true;
    for (int j = 1; j < nblk; j++) starts_out[j] = spec[j].start[v] + d;
    starts_out[nblk] = xe;
    return 1;
}

int gpsb200_carrier_chain(const gpsb200_chan_t *chans, int nblk, int nchan, const double *phase_in,
                          double *phase_out, int threads) {
    if (!chans || !phase_out || nblk < 0 || nchan < 1) return GPSB200_ERR_ARG;
    const double delt = 1.0 / (double) GPSB200_SAMPLERATE;
    auto work = [&](int lo, int hi) {
        for (int c = lo; c < hi; c++) {
            int prn = 0;
            double ph = phase_in ? phase_in[c] : 0.0;
            for (int b = 0; b < nblk; b++) {
                const gpsb200_chan_t &in = chans[(size_t) b * nchan + c];
                if (in.prn <= 0) {
                    prn = 0;
                    continue;
                }
                if ((b == 0 && !phase_in) || in.prn != prn) {
                    if (!(b == 0 && phase_in)) ph = in.carr_phase;
                    prn = in.prn;
                }
                int64_t dummy = 0;
                nco_advance<NCO_CARRIER>(ph, in.f_carr * delt, GPSB200_BLOCK_SAMPLES, dummy);
            }
            phase_out[c] = prn > 0 ? ph : 0.0;
        }
    };
    threads = std::max(1, std::min(threads, nchan));
    std::vector<std::thread> th;
    const int per = (nchan + threads - 1) / threads;
    for (int t = 0; t < threads; t++) {
        const int lo = t * per, hi = std::min(nchan, lo + per);
        if (lo < hi) th.emplace_back(work, lo, hi);
    }
    for (auto &t : th) t.join();
    return GPSB200_OK;
}

int gpsb200_create(const gpsb200_config_t *cfg, gpsb200_ctx_t **out) {
    if (!cfg || !out) return GPSB200_ERR_ARG;
    gpsb200_ctx *ctx = new gpsb200_ctx();
    ctx->cfg = *cfg;
    gpsb200_config_t &c = ctx->cfg;
    if (c.run_samples == 0) c.run_samples = 2400;
    if (c.host_threads <= 0) c.host_threads = (int) std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    if (c.max_nav_frames <= 0) c.max_nav_frames = 1;
    if (c.max_chan < 1 || c.max_chan > GPSB200_MAX_CHAN || c.max_blocks < 1 || c.run_samples < 32 ||
        c.run_samples % 32 != 0 || GPSB200_BLOCK_SAMPLES % c.run_samples != 0 ||
        (c.carrier_nco != GPSB200_CARRIER_FP64 && c.carrier_nco != GPSB200_CARRIER_U32)) {
        delete ctx;
        return GPSB200_ERR_ARG;
    }
    ctx->nruns = GPSB200_BLOCK_SAMPLES / c.run_samples;
    ctx->u32 = c.carrier_nco == GPSB200_CARRIER_U32;
    if (const char *ev = getenv("GPSB200_GRADED_CHUNKS")) ctx->graded_chunks = atoi(ev) != 0;
    ctx->pool.reset(new WorkerPool(std::min(c.host_threads, c.max_chan)));
    *out = ctx;   // from here on errors are reported through the context
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(ctx, GPSB200_ERR_CUDA, "no CUDA device: gpsb200 has no CPU fallback");
    CU(cudaSetDevice(c.device));
    CU(cudaStreamCreateWithFlags(&ctx->s_compute, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
    {   // the pre-phase (latency-bound walk kernels, the lead-in of everything) outranks the synthesis
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(cudaStreamCreateWithPriority(&ctx->s_pre, cudaStreamNonBlocking, hi));
        CU(cudaStreamCreateWithPriority(&ctx->s_ck, cudaStreamNonBlocking, hi));
    }
    for (cudaEvent_t *e : timing_events(ctx)) CU(cudaEventCreate(e));
    const int nchunk = (c.max_blocks + kSynthChunk - 1) / kSynthChunk + (c.max_blocks + kSegBlocks - 1) / kSegBlocks + 5;
    ctx->ev_done.resize(nchunk);
    for (auto &e : ctx->ev_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ctx->max_segs = (c.max_blocks + kSegBlocks - 1) / kSegBlocks + 2;
    ctx->ev_seg.resize(ctx->max_segs);
    for (auto &e : ctx->ev_seg) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU(cudaHostAlloc(&ctx->h_seg_end, (size_t) ctx->max_segs * c.max_chan * sizeof(double), cudaHostAllocMapped));
    CU(cudaHostGetDevicePointer((void **) &ctx->d_seg_end, ctx->h_seg_end, 0));
    ctx->seg_expect.assign((size_t) ctx->max_segs * c.max_chan, -1.0);
    const size_t nbc = (size_t) c.max_blocks * c.max_chan;
    CU(cudaMalloc(&ctx->d_bc, nbc * sizeof(BlockChanDev)));
    CU(cudaHostAlloc(&ctx->h_bc, nbc * sizeof(BlockChanDev), cudaHostAllocDefault));
    CU(cudaMalloc(&ctx->d_ck, nbc * ctx->nruns * sizeof(RunCkpt)));
    CU(cudaHostAlloc(&ctx->h_ck, (size_t) std::min(c.max_blocks, kHostChainBlocks) * c.max_chan * ctx->nruns * sizeof(RunCkpt),
                     cudaHostAllocDefault));
    CU(cudaMalloc(&ctx->d_carr_end, nbc * sizeof(double)));
    CU(cudaMalloc(&ctx->d_atab, (size_t) c.max_blocks * kAtabRows * 32 * sizeof(int32_t)));
    CU(cudaMalloc(&ctx->d_chain_errors, sizeof(int)));
    CU(cudaHostAlloc(&ctx->h_chain_errors, sizeof(int), cudaHostAllocDefault));
    CU(cudaMalloc(&ctx->d_guess, nbc * sizeof(double)));
    CU(cudaHostAlloc(&ctx->h_guess, nbc * sizeof(double), cudaHostAllocDefault));
    ctx->h_guess_abs.assign(nbc, 1);
    ctx->h_span_flags.assign((size_t) ((c.max_blocks + kSpanBlocks - 1) / kSpanBlocks + 1) * c.max_chan, 0);
    CU(cudaMalloc(&ctx->d_carr0, nbc * sizeof(double)));
    CU(cudaHostAlloc(&ctx->h_carr0, nbc * sizeof(double), cudaHostAllocDefault));
    // block probes: one copy in HBM (k_chain reads it), one written by the kernel straight into mapped
    // pinned host memory for the host's block-by-block fallback; span summaries only in mapped host memory
    // (a copy-engine download would queue behind the large result downloads of earlier segments)
    CU(cudaMalloc(&ctx->d_probe, nbc * sizeof(CarrierProbe)));
    CU(cudaHostAlloc(&ctx->h_probe, nbc * sizeof(CarrierProbe), cudaHostAllocMapped));
    CU(cudaHostGetDevicePointer((void **) &ctx->d_probe_host, ctx->h_probe, 0));
    ctx->max_spans = (c.max_blocks + kSpanBlocks - 1) / kSpanBlocks + 1;
    const size_t nsc = (size_t) ctx->max_spans * c.max_chan;
    CU(cudaHostAlloc(&ctx->h_span_sum, nsc * sizeof(CarrierProbe), cudaHostAllocMapped));
    CU(cudaHostGetDevicePointer((void **) &ctx->d_span_sum, ctx->h_span_sum, 0));
    CU(cudaMalloc(&ctx->d_spec, nbc * sizeof(SpanBlockState)));
    if (const char *ev = getenv("GPSB200_TRACE")) ctx->trace_on = atoi(ev) != 0;
    if (const char *ev = getenv("GPSB200_LANES")) ctx->lanes_on = atoi(ev) != 0;
    CU(cudaMalloc(&ctx->d_span_res, nsc * sizeof(SpanRes)));
    CU(cudaHostAlloc(&ctx->h_span_res, nsc * sizeof(SpanRes), cudaHostAllocDefault));
    const size_t navb = (size_t) c.max_nav_frames * c.max_chan * GPSB200_NAV_WORDS * 4;
    CU(cudaMalloc(&ctx->d_nav, navb));
    CU(cudaHostAlloc(&ctx->h_nav, navb, cudaHostAllocDefault));
    memset(ctx->h_nav, 0, navb);
    // packed C/A chips (ca[], gps.c:2817), periodically extended so that any 32-chip window
    // starting at chip 0..1022 is two consecutive words; row = prn
    std::vector<uint32_t> chips((size_t) 33 * kChipWords, 0);
    for (int prn = 1; prn <= 32; prn++) {
        uint8_t ca[GPSB200_CA_LEN];
        ca_code(prn, ca);
        for (int n = 0; n < kChipWords * 32; n++)
            if (ca[n % GPSB200_CA_LEN]) chips[(size_t) prn * kChipWords + (n >> 5)] |= 1u << (n & 31);
    }
    CU(cudaMalloc(&ctx->d_chips, chips.size() * 4));
    CU(cudaMemcpy(ctx->d_chips, chips.data(), chips.size() * 4, cudaMemcpyHostToDevice));
    return GPSB200_OK;
}

void gpsb200_destroy(gpsb200_ctx_t *ctx) {
    if (!ctx) return;
    if (ctx->s_compute) cudaSetDevice(ctx->cfg.device);
    if (ctx->s_compute) cudaStreamSynchronize(ctx->s_compute);
    if (ctx->s_copy) cudaStreamSynchronize(ctx->s_copy);
    if (ctx->s_pre) cudaStreamSynchronize(ctx->s_pre);
    if (ctx->s_ck) cudaStreamSynchronize(ctx->s_ck);
    cudaFree(ctx->d_bc);
    cudaFreeHost(ctx->h_bc);
    cudaFree(ctx->d_ck);
    cudaFreeHost(ctx->h_ck);
    cudaFree(ctx->d_carr_end);
    cudaFree(ctx->d_atab);
    cudaFree(ctx->d_chain_errors);
    cudaFreeHost(ctx->h_chain_errors);
    cudaFree(ctx->d_guess);
    cudaFreeHost(ctx->h_guess);
    cudaFree(ctx->d_carr0);
    cudaFreeHost(ctx->h_carr0);
    cudaFreeHost(ctx->h_probe);
    cudaFree(ctx->d_probe);
    cudaFreeHost(ctx->h_span_sum);
    cudaFree(ctx->d_spec);
    cudaFree(ctx->d_span_res);
    cudaFreeHost(ctx->h_span_res);
    cudaFree(ctx->d_nav);
    cudaFreeHost(ctx->h_nav);
    cudaFree(ctx->d_chips);
    cudaFree(ctx->d_out);
    for (cudaEvent_t *e : timing_events(ctx))
        if (*e) cudaEventDestroy(*e);
    for (auto &e : ctx->ev_done)
        if (e) cudaEventDestroy(e);
    for (auto &e : ctx->ev_seg)
        if (e) cudaEventDestroy(e);
    cudaFreeHost(ctx->h_seg_end);
    if (ctx->s_compute) cudaStreamDestroy(ctx->s_compute);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    if (ctx->s_pre) cudaStreamDestroy(ctx->s_pre);
    if (ctx->s_ck) cudaStreamDestroy(ctx->s_ck);
    delete ctx;
}

int gpsb200_set_nav(gpsb200_ctx_t *ctx, int frame, int chan, const uint32_t dwrd[GPSB200_NAV_WORDS]) {
    if (!ctx || !dwrd) return GPSB200_ERR_ARG;
    if (frame < 0 || frame >= ctx->cfg.max_nav_frames || chan < 0 || chan >= ctx->cfg.max_chan)
        return fail(ctx, GPSB200_ERR_ARG, "gpsb200_set_nav: frame/channel out of range");
    memcpy(ctx->h_nav + ((size_t) frame * ctx->cfg.max_chan + chan) * GPSB200_NAV_WORDS, dwrd, GPSB200_NAV_WORDS * 4);
    ctx->nav_dirty = true;
    return GPSB200_OK;
}

int gpsb200_synth_blocks_device(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan,
                                int sample_size, void *dst_device, void *stream_, double *carr_phase_out,
                                gpsb200_stats_t *stats) {
    int rc = check_call(ctx, chans, nblk, nchan, sample_size, dst_device);
    if (rc) return rc;
    cudaStream_t s = stream_ ? (cudaStream_t) stream_ : ctx->s_compute;
    return run_pipeline(ctx, chans, nblk, nchan, sample_size, dst_device, nullptr, s, nullptr, nullptr, nullptr,
                        carr_phase_out, stats);
}

// ---- time-slice hand-over: one call in three steps (see include/gpsb200.h) --------------------------
int gpsb200_slice_prepare(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size,
                          void *dst_device, void *dst_host, void *stream_, gpsb200_slice_link_t *link) {
    int rc = check_call(ctx, chans, nblk, nchan, sample_size, dst_device ? dst_device : dst_host);
    if (rc) return rc;
    if (!dst_device) {                          // host destination only: stage in the context's own device buffer
        rc = stage_out(ctx, sample_size);
        if (rc) return rc;
        dst_device = ctx->d_out;
    }
    if (!link) return fail(ctx, GPSB200_ERR_ARG, "gpsb200_slice_prepare: link is NULL");
    cudaStream_t s = stream_ ? (cudaStream_t) stream_ : ctx->s_compute;
    cudaStream_t sp = ctx->s_pre;
    CU(cudaEventRecord(ctx->ev_start, s));
    CU(cudaStreamWaitEvent(sp, ctx->ev_start, 0));      // earlier work on s may still read the buffers rewritten now
    CU(cudaStreamWaitEvent(ctx->s_ck, ctx->ev_start, 0));
    rc = upload_nav(ctx, sp);
    if (rc) return rc;
    CU(cudaMemsetAsync(ctx->d_chain_errors, 0, sizeof(int), sp));
    std::vector<ChainState> none(nchan);
    gpsb200_stats_t st{};
    memset(link, 0, sizeof *link);
    rc = drained(ctx, segment_params(ctx, chans, 0, nblk, nchan, sp, none, st, link), s);
    if (rc) return rc;
    ctx->have_last = false;
    ctx->pending.active = true;
    ctx->pending.probed = false;
    ctx->pending.finished = false;
    ctx->pending.nblk = nblk;
    ctx->pending.nchan = nchan;
    ctx->pending.sample_size = sample_size;
    ctx->pending.dst = dst_device;
    ctx->pending.dst_host = dst_host;
    ctx->pending.stream = s;
    ctx->pending.st = st;
    return GPSB200_OK;
}

int gpsb200_slice_probe(gpsb200_ctx_t *ctx, const int32_t *prn_in, const double *phase_guess_in, int eager) {
    if (!ctx) return GPSB200_ERR_ARG;
    if (!ctx->pending.active || ctx->pending.probed)
        return fail(ctx, GPSB200_ERR_ARG, "gpsb200_slice_probe: call gpsb200_slice_prepare first");
    CU(cudaSetDevice(ctx->cfg.device));
    const int nblk = ctx->pending.nblk, nchan = ctx->pending.nchan;
    if (!phases_ok(ctx, nchan, prn_in, phase_guess_in))
        return fail(ctx, GPSB200_ERR_ARG, "gpsb200_slice_probe: phase_guess_in is not a carrier phase of this context");
    ctx->pending.eager = eager != 0;
    const double t0 = now_ms();
    finalize_guesses(ctx, 0, nblk, nchan, prn_in, phase_guess_in);
    ctx->pending.st.host_chain_ms += now_ms() - t0;
    // eager: everything speculative at once, ONE probe and ONE chaining launch over the whole slice (no per-segment
    // tails); lazy: only the first segment's, the others follow one by one in gpsb200_slice_finish
    const int b1 = ctx->pending.eager ? nblk : segments_of(nblk)[0].second;
    const int rc = drained(ctx, speculate(ctx, 0, b1, nchan, ctx->s_pre, ctx->pending.st, true, ctx->ev_seg[0]),
                           ctx->pending.stream);
    if (rc) {
        ctx->pending.active = false;
        return rc;
    }
    ctx->pending.probed = true;
    return GPSB200_OK;
}

namespace {
int slice_finish_inner(gpsb200_ctx *ctx, std::vector<ChainState> &chain, gpsb200_stats_t &st, int32_t *prn_out,
                       double *phase_out, gpsb200_handoff_fn handoff, void *user) {
    const int nblk = ctx->pending.nblk, nchan = ctx->pending.nchan, sample_size = ctx->pending.sample_size;
    cudaStream_t s = ctx->pending.stream, sk = ctx->s_ck;
    const auto segs = segments_of(nblk);
    const int nseg = (int) segs.size();
    std::vector<int64_t> slow(nseg, 0);
    std::vector<std::vector<ChainState>> after(nseg);
    bool eager = ctx->pending.eager;
    ctx->trace_t0 = now_ms();
    trace(ctx, "slice_finish");
    if (ctx->u32) {
        // The exact incoming state is known now: rebase the prepared start phases on it. The outgoing state is then a
        // closed form, so it is handed over at once (eager order).
        std::vector<int32_t> pi(nchan);
        std::vector<double> xi(nchan);
        export_chain(chain, nchan, pi.data(), xi.data());
        CU(cudaStreamSynchronize(ctx->s_pre));       // the prepare pass's parameter upload has read h_bc
        u32_rebase(ctx, nblk, nchan, pi.data(), xi.data());
        CU(cudaMemcpyAsync(ctx->d_bc, ctx->h_bc, (size_t) nblk * nchan * sizeof(BlockChanDev), cudaMemcpyHostToDevice, sk));
        st.h2d_bytes += (int64_t) ((size_t) nblk * nchan * sizeof(BlockChanDev));
        eager = true;
    }
    int rc = GPSB200_OK;
    if (eager) {
        // A successor waits for the outgoing state: scan EVERYTHING first (all probes were submitted up front), hand
        // the exact state on, and only then enqueue the long kernels -- a message sent behind them would wait for them.
        for (int i = 0; i < nseg; i++) {
            rc = scan(ctx, segs[i].first, segs[i].second, nchan, chain, st, ctx->ev_seg[0], slow[i]);
            if (rc) return rc;
            after[i] = chain;
        }
        trace(ctx, "host scan done");
        export_chain(chain, nchan, prn_out, phase_out);
        if (handoff) handoff(user, prn_out, phase_out);
        trace(ctx, "handed over");
    }
    for (int i = 0, ichunk = 0; i < nseg; i++) {
        const int b0 = segs[i].first, b1 = segs[i].second;
        if (!eager) {
            // lazy: host scan of this segment as soon as ITS probes are done; checkpoints on a stream of their own
            rc = scan(ctx, b0, b1, nchan, chain, st, ctx->ev_seg[i], slow[i]);
            if (rc) return rc;
            after[i] = chain;
        }
        rc = checkpoints(ctx, b0, b1, nchan, sk, st, i == 0, slow[i], i, after[i]);
        if (!rc) rc = synthesize(ctx, b0, b1, nchan, sample_size, ctx->pending.dst, ctx->pending.dst_host, sk, s, st, ichunk);
        if (rc) return rc;
        if (!eager && b1 < nblk) {
            // lazy: the next segment's speculative work is submitted only now, BEHIND this segment's synthesis, from
            // guesses re-anchored on the exact state just resolved
            const int n1 = std::min(nblk, b1 + kSegBlocks);
            reanchor_guesses(ctx, b1, n1, nchan, chain);
            rc = speculate(ctx, b1, n1, nchan, ctx->s_pre, st, false, ctx->ev_seg[i + 1]);
            if (rc) return rc;
        }
    }
    if (!eager) {
        export_chain(chain, nchan, prn_out, phase_out);
        if (handoff) handoff(user, prn_out, phase_out);
    }
    ctx->pending.nseg = nseg;
    CU(cudaEventRecord(ctx->ev_end, s));
    CU(cudaMemcpyAsync(ctx->h_chain_errors, ctx->d_chain_errors, sizeof(int), cudaMemcpyDeviceToHost, sk));
    trace(ctx, "checkpoints + synthesis enqueued");
    return GPSB200_OK;
}
}  // namespace

int gpsb200_slice_finish_cb(gpsb200_ctx_t *ctx, const int32_t *prn_in, const double *phase_in, int32_t *prn_out,
                            double *phase_out, gpsb200_stats_t *stats, gpsb200_handoff_fn handoff, void *user) {
    if (!ctx) return GPSB200_ERR_ARG;
    if (!ctx->pending.active || !ctx->pending.probed)
        return fail(ctx, GPSB200_ERR_ARG, "gpsb200_slice_finish: call gpsb200_slice_prepare and gpsb200_slice_probe first");
    CU(cudaSetDevice(ctx->cfg.device));
    const int nblk = ctx->pending.nblk, nchan = ctx->pending.nchan;
    if (!phases_ok(ctx, nchan, prn_in, phase_in))
        return fail(ctx, GPSB200_ERR_ARG, "gpsb200_slice_finish: phase_in is not a carrier phase of this context");
    ctx->pending.active = false;
    std::vector<ChainState> chain(nchan);
    seed_chain(chain, nchan, prn_in, phase_in);
    gpsb200_stats_t st = ctx->pending.st;
    std::vector<int32_t> po(nchan, 0);
    std::vector<double> xo(nchan, 0.0);
    const int rc =
        drained(ctx, slice_finish_inner(ctx, chain, st, po.data(), xo.data(), handoff, user), ctx->pending.stream);
    if (rc) return rc;
    ctx->last = args_of(ctx, 0, nblk, nchan, ctx->pending.sample_size, ctx->pending.dst);
    ctx->have_last = true;
    ctx->pending.finished = true;
    for (int c = 0; c < nchan; c++) {
        if (prn_out) prn_out[c] = po[c];
        if (phase_out) phase_out[c] = xo[c];
    }
    if (stats) *stats = st;
    return GPSB200_OK;
}

int gpsb200_slice_finish(gpsb200_ctx_t *ctx, const int32_t *prn_in, const double *phase_in, int32_t *prn_out,
                         double *phase_out, gpsb200_stats_t *stats) {
    return gpsb200_slice_finish_cb(ctx, prn_in, phase_in, prn_out, phase_out, stats, nullptr, nullptr);
}

int gpsb200_slice_wait(gpsb200_ctx_t *ctx) {
    if (!ctx || !ctx->s_compute) return GPSB200_ERR_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    CU(cudaStreamSynchronize(ctx->s_pre));
    CU(cudaStreamSynchronize(ctx->s_ck));
    if (ctx->pending.stream) CU(cudaStreamSynchronize(ctx->pending.stream));
    CU(cudaStreamSynchronize(ctx->s_copy));
    if (ctx->pending.finished) {
        ctx->pending.finished = false;
        return verify_chain(ctx, ctx->pending.nseg, ctx->pending.nchan);
    }
    return GPSB200_OK;
}

int gpsb200_slice_link_host(const gpsb200_chan_t *chans, int nblk, int nchan, gpsb200_slice_link_t *link) {
    // the link of a slice from its parameters alone (what gpsb200_slice_prepare also returns); no device involved
    if (!chans || !link || nblk < 1 || nchan < 1 || nchan > GPSB200_MAX_CHAN) return GPSB200_ERR_ARG;
    const double delt = 1.0 / (double) GPSB200_SAMPLERATE;
    memset(link, 0, sizeof *link);
    for (int c = 0; c < nchan; c++) {
        long double acc = 0.0L;
        int prev = chans[c].prn;
        bool absolute = false;
        link->prn_first[c] = prev;
        link->first_phase[c] = prev > 0 ? chans[c].carr_phase : 0.0;
        for (int b = 0; b < nblk; b++) {
            const gpsb200_chan_t &in = chans[(size_t) b * nchan + c];
            if (in.prn <= 0) {
                prev = 0;
                absolute = true;
                continue;
            }
            if (in.prn != prev) {
                acc = in.carr_phase;
                absolute = true;
            }
            prev = in.prn;
            const double cc = in.f_carr * delt;
            acc += (long double) GPSB200_BLOCK_SAMPLES * ((long double) cc + (long double) carrier_drift_per_step(cc));
            acc -= floorl(acc);
        }
        link->prn_last[c] = prev > 0 ? prev : 0;
        link->reset_inside[c] = absolute ? 1 : 0;
        const double g = (double) acc;
        link->value[c] = (g >= 0.0 && g < 1.0) ? g : 0.0;
    }
    return GPSB200_OK;
}

int gpsb200_link_apply(const gpsb200_slice_link_t *link, int nchan, const int32_t *prn_in, const double *phase_in,
                       int32_t *prn_out, double *phase_out) {
    if (!link || !prn_out || !phase_out || nchan < 1 || nchan > GPSB200_MAX_CHAN) return GPSB200_ERR_ARG;
    for (int c = 0; c < nchan; c++) {
        if (link->prn_last[c] <= 0) {
            prn_out[c] = 0;
            phase_out[c] = 0.0;
            continue;
        }
        double ph = link->value[c];
        if (!link->reset_inside[c]) {
            const bool cont = prn_in && phase_in && prn_in[c] > 0 && prn_in[c] == link->prn_first[c];
            ph += cont ? phase_in[c] : link->first_phase[c];
            if (ph >= 1.0) ph -= 1.0;
        }
        prn_out[c] = link->prn_last[c];
        phase_out[c] = (ph >= 0.0 && ph < 1.0) ? ph : 0.0;
    }
    return GPSB200_OK;
}

int gpsb200_slice_link_host_nco(const gpsb200_chan_t *chans, int nblk, int nchan, int carrier_nco,
                                gpsb200_slice_link_t *link) {
    if (carrier_nco == GPSB200_CARRIER_FP64) return gpsb200_slice_link_host(chans, nblk, nchan, link);
    if (carrier_nco != GPSB200_CARRIER_U32 || !chans || !link || nblk < 1 || nchan < 1 || nchan > GPSB200_MAX_CHAN)
        return GPSB200_ERR_ARG;
    // exact: the advance of a block is 300000 * carr_phasestep modulo 2^32 (gps.c:2828)
    memset(link, 0, sizeof *link);
    for (int c = 0; c < nchan; c++) {
        uint32_t acc = 0u;
        int prev = chans[c].prn;
        bool absolute = false;
        link->prn_first[c] = prev;
        link->first_phase[c] = prev > 0 ? chans[c].carr_phase : 0.0;
        for (int b = 0; b < nblk; b++) {
            const gpsb200_chan_t &in = chans[(size_t) b * nchan + c];
            if (in.prn <= 0) {
                prev = 0;
                absolute = true;
                continue;
            }
            if (in.prn != prev) {
                if (!valid_u32_phase(in.carr_phase)) return GPSB200_ERR_ARG;
                acc = (uint32_t) in.carr_phase;
                absolute = true;
            }
            prev = in.prn;
            acc += (uint32_t) GPSB200_BLOCK_SAMPLES * (uint32_t) lanes::u32_carrier_step(in.f_carr);
        }
        link->prn_last[c] = prev > 0 ? prev : 0;
        link->reset_inside[c] = absolute ? 1 : 0;
        link->value[c] = (double) acc;
    }
    return GPSB200_OK;
}

int gpsb200_link_apply_nco(const gpsb200_slice_link_t *link, int nchan, int carrier_nco, const int32_t *prn_in,
                           const double *phase_in, int32_t *prn_out, double *phase_out) {
    if (carrier_nco == GPSB200_CARRIER_FP64) return gpsb200_link_apply(link, nchan, prn_in, phase_in, prn_out, phase_out);
    if (carrier_nco != GPSB200_CARRIER_U32 || !link || !prn_out || !phase_out || nchan < 1 || nchan > GPSB200_MAX_CHAN)
        return GPSB200_ERR_ARG;
    for (int c = 0; c < nchan; c++) {
        if (link->prn_last[c] <= 0) {
            prn_out[c] = 0;
            phase_out[c] = 0.0;
            continue;
        }
        uint32_t u = (uint32_t) link->value[c];
        if (!link->reset_inside[c]) {
            const bool cont = prn_in && phase_in && prn_in[c] > 0 && prn_in[c] == link->prn_first[c];
            const double base = cont ? phase_in[c] : link->first_phase[c];
            if (!valid_u32_phase(base)) return GPSB200_ERR_ARG;
            u += (uint32_t) base;
        }
        prn_out[c] = link->prn_last[c];
        phase_out[c] = (double) u;
    }
    return GPSB200_OK;
}

const char *gpsb200_synth_kernel_name(const gpsb200_ctx_t *ctx, int nchan) {
    if (!ctx) return "";
    SynthArgs a{};
    a.nchan = nchan;
    a.run_samples = ctx->cfg.run_samples;
    a.lanes = ctx->lanes_on && !ctx->lanes_veto ? 1 : 0;
    if (ctx->u32) return synth_lanes_applicable(a) ? "k_synth_lanes_u32" : "k_synth_u32";
    return synth_lanes_applicable(a) ? "k_synth_lanes" : "k_synth";
}

int gpsb200_debug_corrupt_chain(gpsb200_ctx_t *ctx, int on) {
    if (!ctx) return GPSB200_ERR_ARG;
    if (ctx->u32) return fail(ctx, GPSB200_ERR_ARG, "gpsb200_debug_corrupt_chain: a U32 carrier context has no carrier chain");
    ctx->fault_inject_chain = on != 0;
    return GPSB200_OK;
}

int gpsb200_carrier_chain_device(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan,
                                 const double *phase_in, double *phase_out) {
    if (!ctx || !chans || !phase_out || nblk < 0 || nchan < 1 || nchan > ctx->cfg.max_chan) return GPSB200_ERR_ARG;
    if (!ctx->s_compute) return fail(ctx, GPSB200_ERR_CUDA, "context has no CUDA device");
    if (ctx->pending.active) return fail(ctx, GPSB200_ERR_ARG, "a call begun with gpsb200_slice_prepare has not been finished");
    CU(cudaSetDevice(ctx->cfg.device));
    cudaStream_t s = ctx->s_compute;
    std::vector<ChainState> chain(nchan);
    gpsb200_stats_t st{};        // (not reported)
    if (phase_in && nblk > 0)
        for (int c = 0; c < nchan; c++)
            if (chans[c].prn > 0) {
                if (ctx->u32 && !valid_u32_phase(phase_in[c])) return fail(ctx, GPSB200_ERR_ARG, "phase_in: not a u32 phase");
                chain[c].prn = chans[c].prn;
                chain[c].phase = phase_in[c];
            }
    for (int w0 = 0; w0 < nblk; w0 += ctx->cfg.max_blocks) {
        const int nw = std::min(ctx->cfg.max_blocks, nblk - w0);
        const gpsb200_chan_t *cw = chans + (size_t) w0 * nchan;
        int rc = prepare_blocks(ctx, cw, 0, nw, nchan, chain);
        if (rc) return rc;
        if (!ctx->u32)              // the probes read the records (a U32 chain is a closed form of them: no device work)
            CU(cudaMemcpyAsync(ctx->d_bc, ctx->h_bc, (size_t) nw * nchan * sizeof(BlockChanDev), cudaMemcpyHostToDevice, s));
        int64_t slow = 0;
        rc = speculate(ctx, 0, nw, nchan, s, st, false, ctx->ev_seg[0]);
        if (!rc) rc = scan(ctx, 0, nw, nchan, chain, st, ctx->ev_seg[0], slow);
        if (rc) return rc;
    }
    ctx->have_last = false;
    for (int c = 0; c < nchan; c++) phase_out[c] = chain[c].prn > 0 ? chain[c].phase : 0.0;
    return GPSB200_OK;
}

int gpsb200_replay_device(gpsb200_ctx_t *ctx, void *dst_device, void *stream_, int kernel_mask) {
    if (!ctx || !ctx->have_last) return GPSB200_ERR_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    cudaStream_t s = stream_ ? (cudaStream_t) stream_ : ctx->s_compute;
    SynthArgs a = ctx->last;
    if (dst_device) a.out = dst_device;
    if (kernel_mask & 8) CU(launch_tables(a, s));
    if ((kernel_mask & 4) && !ctx->u32) {       // a U32 call has no probes to replay
        CU(launch_probe(a, s));
        CU(launch_chain(a, s));
    }
    if (kernel_mask & 1) CU(launch_checkpoints(a, s));
    if (kernel_mask & 2) CU(launch_synth(a, s));
    return GPSB200_OK;
}

int gpsb200_synth_blocks_scatter(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size,
                                 void *const *dst_blocks, double *carr_phase_out, gpsb200_stats_t *stats) {
    if (!ctx || !dst_blocks) return GPSB200_ERR_ARG;
    for (int b = 0; b < nblk; b++)
        if (!dst_blocks[b]) return fail(ctx, GPSB200_ERR_ARG, "gpsb200_synth_blocks_scatter: NULL block destination");
    ctx->scatter = dst_blocks;
    const int rc = gpsb200_synth_blocks(ctx, chans, nblk, nchan, sample_size, dst_blocks[0], carr_phase_out, stats);
    ctx->scatter = nullptr;
    return rc;
}

int gpsb200_synth_blocks(gpsb200_ctx_t *ctx, const gpsb200_chan_t *chans, int nblk, int nchan, int sample_size,
                         void *dst, double *carr_phase_out, gpsb200_stats_t *stats) {
    int rc = check_call(ctx, chans, nblk, nchan, sample_size, dst);
    if (rc) return rc;
    rc = stage_out(ctx, sample_size);
    if (rc) return rc;
    return run_pipeline(ctx, chans, nblk, nchan, sample_size, ctx->d_out, dst, ctx->s_compute, nullptr, nullptr, nullptr,
                        carr_phase_out, stats);
}

}  // extern "C"
