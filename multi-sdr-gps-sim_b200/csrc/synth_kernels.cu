// sm_100a kernels for the GPS L1 C/A sample loop of multi-sdr-gps-sim
// (reference: gps.c:2767-2857). No tensor cores: the path is a per-sample
// NCO + table lookup + integer accumulate; the bound is instruction issue and
// shared-memory wavefronts, the output is 2 (int8) or 4 (int16) bytes per sample.
//
// Work decomposition
//   block  = 0.1 s = 300000 samples (the reference's unit, sdr.h:26)
//   run    = run_samples consecutive samples of one block (default 2400)
//   k_probe       : one thread per (block, channel) walks the carrier NCO through the
//                   block from a GUESSED start phase (speculative, parallel in time);
//                   the host turns the probes into exact start phases (nco_exact.h).
//   k_tables      : one thread per (block, carrier-table row < 256, lane column): the gain-scaled
//                   carrier table of every block, written once to HBM; k_synth's CTAs (several
//                   per block) fetch it with one TMA bulk copy each instead of recomputing it.
//   k_checkpoints : two threads per (block, channel) walk the code and the carrier NCO
//                   through the block with the exact O(#binade crossings) fast-forward
//                   and store the state at every run start.
//   k_synth       : one warp per run (32 channels) or per 2/4 runs (<=16/<=8
//                   channels). LANE = CHANNEL: every lane steps its channel's two
//                   FP64 NCOs sample by sample with the reference's own rounding
//                   (__dadd_rn), looks up the gain-scaled carrier table and the
//                   chip sign (from a per-lane register window of the packed C/A code),
//                   and the warp adds the channels with one REDUX.SUM (packed
//                   I + Q<<16). Sums are staged in shared memory and written out 64
//                   samples at a time as coalesced int8/int16 I/Q.
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "nco_exact.h"
#include "synth_kernels.h"
#include "synth_tables.h"

namespace gpsb200 {

__constant__ uint8_t c_quarter_sine[128] = {GPSB200_QUARTER_SINE};

__device__ __forceinline__ int sine512(int k) {
    k &= 511;
    const int q = k & 255;
    const int v = c_quarter_sine[q < 128 ? q : 255 - q];
    return k < 256 ? v : -v;
}

static int group_for(int nchan) { return nchan > 16 ? 32 : (nchan > 8 ? 16 : 8); }

// ---------------------------------------------------------------------------------
// Carrier tables: atab[block][k][lane] = I + (Q << 16) with I = (int)(cosTable512[k] * gain),
// Q = (int)(sinTable512[k] * gain) of the lane's channel (gps.c:2781-2782: int product ->
// double, ONE rounding by the multiply, truncation toward zero). Rows k and k + 256 are
// negatives of each other (sin[k + 256] = -sin[k], truncation is sign-symmetric), so one
// thread writes both. Columns repeat with the lane group size (lane = channel + GROUP * j).
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_tables(SynthArgs a, int group) {
    const long idx = (long) blockIdx.x * blockDim.x + threadIdx.x;
    const long per_blk = 256L * 32;
    const int b = (int) (idx / per_blk);
    if (b >= a.nblk) return;
    const int rem = (int) (idx - (long) b * per_blk), k = rem >> 5, col = rem & 31, c = col % group;
    const BlockChanDev *bc = a.bc + (size_t) b * a.nchan;
    int32_t e = 0;
    if (c < a.nchan && bc[c].prn > 0) {
        const double gain = bc[c].gain;
        const int ai = __double2int_rz(__dmul_rn((double) sine512(k + 128), gain));
        const int aq = __double2int_rz(__dmul_rn((double) sine512(k), gain));
        e = ai + aq * 65536;
    }
    int32_t *t = a.atab + (size_t) b * kAtabRows * 32 + col;
    t[k * 32] = e;
    t[(k + 256) * 32] = -e;
    if (k == 255) t[512 * 32] = -e;                 // guard row 512 = row 511
}

// ---------------------------------------------------------------------------------
// Carrier probe and checkpoint kernels
// ---------------------------------------------------------------------------------
// Thread mapping of both: warp = 32 consecutive blocks of ONE channel (same satellite,
// similar Doppler, hence similar iteration counts across the lanes of a warp).
__device__ __forceinline__ bool map_block_chan(const SynthArgs &a, int idx, int &b, int &c) {
    const int nblk_pad = (a.nblk + 31) & ~31;
    c = idx / nblk_pad;
    b = idx - c * nblk_pad;
    return c < a.nchan && b < a.nblk;
}

__global__ void __launch_bounds__(128) k_probe(SynthArgs a) {
    // two threads per (block, channel): one per parity variant (nco_exact.h); a warp is 32 consecutive
    // blocks of one channel
    const int nblk_pad = (a.nblk + 31) & ~31;
    const int per_v = nblk_pad * a.nchan;
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int v = idx / per_v;
    idx -= v * per_v;
    int b, c;
    if (v > 1 || !map_block_chan(a, idx, b, c)) return;
    const size_t i = (size_t) b * a.nchan + c;
    const BlockChanDev p = a.bc[i];
    CarrierProbe o;
    if (p.prn > 0) {
        carrier_probe_variant(a.guess[i], p.c_carr, kBlockSamples, v, o);
    } else {
        o.n_w = -1;
        o.x_w = 0.0;
        o.x_end[v] = o.m_pos[v] = o.m_neg[v] = 0.0;
    }
    // two copies: HBM for k_chain, mapped host memory for the host's (rare) block-by-block fallback
    CarrierProbe *dsts[2] = {a.probe + i, a.probe_host ? a.probe_host + i : nullptr};
#pragma unroll
    for (int k = 0; k < 2; k++) {
        CarrierProbe *dst = dsts[k];
        if (!dst) continue;
        if (v == 0) {
            dst->x_w = o.x_w;
            dst->n_w = o.n_w;
            dst->pad = 0;
        }
        dst->x_end[v] = o.x_end[v];
        dst->m_pos[v] = o.m_pos[v];
        dst->m_neg[v] = o.m_neg[v];
    }
}

struct ColumnParams {
    const BlockChanDev *col;
    int nchan;
    __device__ __forceinline__ void operator()(int j, double &cc, int32_t &prn) const {
        const BlockChanDev &p = col[(size_t) j * nchan];
        cc = p.c_carr;
        prn = p.prn;
    }
};

// One thread per (span, channel, parity variant): chain the span's block probes speculatively from the span's
// guessed start phase (nco_exact.h: span_chain). Serial over the span's blocks, a few walk iterations each.
__global__ void __launch_bounds__(64) k_chain(SynthArgs a) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int per_v = a.nspan * a.nchan;
    const int V = idx / per_v;
    idx -= V * per_v;
    if (V > 1) return;
    const int sp = idx / a.nchan, c = idx - sp * a.nchan;
    const int b0 = sp * a.span_blocks, nb = min(a.span_blocks, a.nblk - b0);
    const size_t i0 = (size_t) b0 * a.nchan + c;
    CarrierProbe sum;
    bool ok;
    const ColumnParams col{a.bc + i0, a.nchan};   // this channel's column: block j at bc[j * nchan]
    span_chain(a.probe + i0, col, nb, (size_t) a.nchan, a.guess[i0], V, sum, ok, a.spec + i0);
    CarrierProbe *dst = a.span_sum + (size_t) sp * a.nchan + c;
    if (V == 0) {
        dst->x_w = sum.x_w;
        dst->n_w = sum.n_w;
        dst->pad = 0;
    }
    dst->x_end[V] = sum.x_end[V];
    dst->m_pos[V] = ok ? sum.m_pos[V] : 0.0;
    dst->m_neg[V] = ok ? sum.m_neg[V] : 0.0;
}

// exact carrier phase at the first sample of block b of channel c, as the host scan resolved it
__device__ __forceinline__ double resolved_start(const SynthArgs &a, int b, int c) {
    const int sp = b / a.span_blocks;
    const SpanRes r = a.span_res[(size_t) sp * a.nchan + c];
    if (r.mode == 1) return a.carr0[(size_t) b * a.nchan + c];
    if (r.mode == 2) return 0.0;
    if (b == sp * a.span_blocks) return r.start;
    return a.spec[(size_t) b * a.nchan + c].start[r.variant] + r.shift;     // exact: see span_chain()
}

__global__ void __launch_bounds__(128) k_checkpoints(SynthArgs a) {
    // role 0: one thread per (block, channel) walks the code NCO (+ NAV position) through the block;
    // role 1: one thread per (block, channel) walks the carrier through the block from its resolved start
    const int nblk_pad = (a.nblk + 31) & ~31;
    const int per_code = nblk_pad * a.nchan;
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int b, c;
    if (idx < per_code) {
        if (!map_block_chan(a, idx, b, c)) return;
        const size_t i = (size_t) b * a.nchan + c;
        const BlockChanDev p = a.bc[i];
        RunCkpt *ck = a.ck + (size_t) b * a.nruns * a.nchan + c;
        double y = p.code0;
        int iword = p.nav0 & 0xFF, ibit = (p.nav0 >> 8) & 0xFF, icode = (p.nav0 >> 16) & 0xFF;
        const uint32_t step = (uint32_t) p.step_u32;
        for (int r = 0; r < a.nruns; r++) {
            RunCkpt *o = ck + (size_t) r * a.nchan;
            o->y = y;
            o->nav = (uint32_t) iword | ((uint32_t) ibit << 8) | ((uint32_t) icode << 16);
            o->pad = 0;
            // U32 carrier (gps.c:2828): exact closed form, modulo 2^32
            if (a.u32) o->x = p.prn > 0 ? (double) (p.u0 + (uint32_t) (r * a.run_samples) * step) : 0.0;
            if (p.prn <= 0) continue;
            int64_t periods = 0;
            nco_advance<NCO_CODE>(y, p.c_code, a.run_samples, periods);
            nav_advance(iword, ibit, icode, periods);
        }
        if (a.u32) {
            const double x_end = p.prn > 0 ? (double) (p.u0 + (uint32_t) kBlockSamples * step) : 0.0;
            if (a.carr_end) a.carr_end[i] = x_end;
            if (a.last_end_host && b == a.nblk - 1) a.last_end_host[c] = x_end;
        }
        return;
    }
    if (a.u32) return;          // the grid is rounded up to whole CTAs: U32 launches have no carrier threads
    idx -= per_code;
    if (!map_block_chan(a, idx, b, c)) return;
    const size_t i = (size_t) b * a.nchan + c;
    const BlockChanDev p = a.bc[i];
    RunCkpt *ck = a.ck + (size_t) b * a.nruns * a.nchan + c;
    double x = 0.0;
    if (p.prn > 0) {
        // exact walk of the whole block from its resolved start, storing every run start
        x = resolved_start(a, b, c);
        for (int r = 0; r < a.nruns; r++) {
            ck[(size_t) r * a.nchan].x = x;
            int64_t dummy = 0;
            nco_advance<NCO_CARRIER>(x, p.c_carr, a.run_samples, dummy);
        }
        // ... whose end must BE the start phase resolved for the next block of the same satellite in this launch
        if (b + 1 < a.nblk && a.bc[i + a.nchan].prn == p.prn && f64_bits(resolved_start(a, b + 1, c)) != f64_bits(x) &&
            a.chain_errors)
            atomicAdd(a.chain_errors, 1);
    } else {
        for (int r = 0; r < a.nruns; r++) ck[(size_t) r * a.nchan].x = 0.0;
    }
    if (a.carr_end) a.carr_end[i] = x;
    if (a.last_end_host && b == a.nblk - 1) a.last_end_host[c] = x;
}

// ---------------------------------------------------------------------------------
// Synthesis kernel
// ---------------------------------------------------------------------------------
constexpr int kMaxWarps = 24;
constexpr int kChunkMax = 64;           // samples per chunk (chip window refill / output flush)

template <int GROUP>
struct SynthSmem {
    int32_t atab[kAtabRows][32];                 // [k][lane]: I + (Q << 16), gain-scaled (gps.c:2781-2782)
    uint32_t cabits[kChipWords][GROUP];          // [word][channel]: C/A chips, bit n = ca[n mod 1023], n < 1056
    uint32_t nav[kNavWords][GROUP];              // NAV words of this block's frame
    alignas(16) int32_t stage[kMaxWarps][kChunkMax * (32 / GROUP)];
    alignas(8) uint64_t bar;                     // mbarrier of the carrier-table bulk copy // per-warp staging of one chunk of samples per run
};

template <int GROUP>
__device__ __forceinline__ int group_sum(int v) {
    if (GROUP == 32) {
        return __reduce_add_sync(0xFFFFFFFFu, v);
    } else {
#pragma unroll
        for (int off = GROUP / 2; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
        return v;
    }
}

// U32: the reference's integer carrier build (gps.c:2777, 2828): the carrier is a u32 add per sample and the index
// (u >> 16) & 511 -- no FP64 carrier, no carrier wrap test; the code NCO, NAV bits and the channel sum are unchanged.
template <int GROUP, bool IQ16, bool U32>
__global__ void __launch_bounds__(kMaxWarps * 32, 2) k_synth(SynthArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SynthSmem<GROUP> &sm = *reinterpret_cast<SynthSmem<GROUP> *>(smem_raw);
    constexpr int RPW = 32 / GROUP;               // runs per warp

    const int b = blockIdx.x / a.ctas_per_block;
    const int g = blockIdx.x - b * a.ctas_per_block;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int ch = lane % GROUP, sub = lane / GROUP;
    const BlockChanDev *bc = a.bc + (size_t) b * a.nchan;

    // ---- per-CTA tables ----------------------------------------------------------
    // carrier table of this block: one TMA bulk copy global -> shared, completion on an mbarrier;
    // the small tables are gathered by the threads meanwhile
    const uint32_t bar = (uint32_t) __cvta_generic_to_shared(&sm.bar);
    constexpr uint32_t kAtabBytes = kAtabRows * 32 * 4;
    static_assert(kAtabBytes % 16 == 0, "bulk copy size");
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(1) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        const int32_t *src = a.atab + (size_t) b * kAtabRows * 32;
        const uint32_t dst = (uint32_t) __cvta_generic_to_shared(&sm.atab[0][0]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(kAtabBytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                     "l"(src), "r"(kAtabBytes), "r"(bar)
                     : "memory");
    }
    for (int i = tid; i < kChipWords * GROUP; i += nthr) {
        const int w = i / GROUP, c = i % GROUP;
        uint32_t v = 0;
        if (c < a.nchan && bc[c].prn > 0) v = a.chipbits[bc[c].prn * kChipWords + w];
        sm.cabits[w][c] = v;
    }
    for (int i = tid; i < kNavWords * GROUP; i += nthr) {
        const int w = i / GROUP, c = i % GROUP;
        uint32_t v = 0;
        if (c < a.nchan && bc[c].prn > 0)
            v = a.nav[((size_t) bc[c].frame * a.nav_stride + c) * kNavWords + w];
        sm.nav[w][c] = v;
    }
    {
        uint32_t done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.b32 %0, 1, 0, p; }"
                         : "=r"(done)
                         : "r"(bar), "r"(0)
                         : "memory");
    }
    __syncthreads();

    // ---- this lane's run and channel ------------------------------------------------
    const int run_first = g * a.runs_per_cta;
    const int run_last = min(run_first + a.runs_per_cta, a.nruns);
    const int r = run_first + warp * RPW + sub;
    const bool run_ok = r < run_last;
    const bool active = run_ok && ch < a.nchan && bc[ch].prn > 0;
    if (__ballot_sync(0xFFFFFFFFu, run_ok) == 0) return;

    double x = 0.0, y = 0.0, cc = 0.0, dd = 0.0;
    uint32_t u = 0u, us = 0u;                                 // U32 carrier: phase, step
    int iword = 0, ibit = 0, icode = 0;
    if (active) {
        const RunCkpt k0 = a.ck[((size_t) b * a.nruns + r) * a.nchan + ch];
        if (U32) {
            u = (uint32_t) k0.x;
            us = (uint32_t) bc[ch].step_u32;
        } else {
            x = k0.x;
        }
        y = k0.y;
        iword = k0.nav & 0xFF;
        ibit = (k0.nav >> 8) & 0xFF;
        icode = (k0.nav >> 16) & 0xFF;
        if (!U32) cc = bc[ch].c_carr;                         // U32: cc = 0, the FP64 carrier never runs
        dd = bc[ch].c_code;
    }
    // floor(x*512) and floor(y) come out of the low mantissa word of a round-toward-zero
    // add of 2^43 / 2^52 (exact: the addend is an integer-valued double).
    const double K43 = 8796093022208.0;
    const double K52 = 4503599627370496.0;
    auto nav_bit = [&](int iw, int ib) -> int {
        const uint32_t w = sm.nav[iw < kNavWords ? iw : kNavWords - 1][ch];
        return (w >> (29 - ib)) & 1;                          // gps.c:2812
    };
    int dbit = nav_bit(iword, ibit);
    // Conservative 8-step look-ahead (see below): 8 steps move a phase by at most 8*(|c| + ulp/2):
    // carrier (phase < 1, ulp <= 2^-53): 8*|c| + 2^-51, covered by 8*|c| + 2^-50; code (phase < 1024,
    // ulp <= 2^-43): 8*d + 2^-41, covered by 8*d + 2^-40. "phase + that can leave the range" is tested on
    // the high words only (monotone for positive doubles), which can only err towards "at risk" -- by up
    // to 2^-20 relative, far more than any rounding of the thresholds themselves.
    const double cc9 = 8.0 * fabs(cc) + 0x1p-50, dd9 = 8.0 * dd + 0x1p-40;
    int thr_x_hi = 0x7FFFFFFF, thr_x_lo = -1;                  // cc == 0: never at risk
    if (cc > 0.0) thr_x_hi = cc9 < 1.0 ? __double2hiint(1.0 - cc9) : 0;
    if (cc < 0.0) thr_x_lo = __double2hiint(cc9);
    const int thr_y = dd9 < 1023.0 ? __double2hiint(1023.0 - dd9) : 0;
    int32_t *stage = &sm.stage[warp][0];
    // shared-window byte address of this lane's column of the carrier table
    const uint32_t abase = (uint32_t) __cvta_generic_to_shared(&sm.atab[0][lane]);
    const uint32_t *ccol = &sm.cabits[0][ch];

    // ---- quantise + pack LEN samples per run (gps.c:2833-2845) ----------------------------
    // lane (sub, ch) converts SPL = LEN / GROUP consecutive samples of its run: contiguous bytes
    auto flush = [&](auto len_tag, int s0) {
        constexpr int LEN = decltype(len_tag)::value;
        constexpr int SPL = LEN / GROUP;
        if (!run_ok) return;
        const size_t samp0 = (size_t) b * kBlockSamples + (size_t) r * a.run_samples + (size_t) s0 + ch * SPL;
        uint32_t w[SPL];                                       // int16: one word per sample; int8: two samples per word
#pragma unroll
        for (int t = 0; t < SPL; t++) {
            const int p = stage[sub * kChunkMax + ch * SPL + t];
            const int iv = (int) (short) (p & 0xFFFF);         // (short) i_acc, gps.c:2834
            const int qv = (p - iv) >> 16;                     // (short) q_acc, gps.c:2835
            if (IQ16) {
                w[t] = ((uint32_t) iv & 0xFFFFu) | ((uint32_t) qv << 16);
            } else {
                const uint32_t two = (((uint32_t) (iv >> 4)) & 0xFFu) | ((((uint32_t) (qv >> 4)) & 0xFFu) << 8);  // gps.c:2844
                if (t & 1) w[t >> 1] |= two << 16;
                else w[t >> 1] = two;
            }
        }
        constexpr int NBYTES = SPL * (IQ16 ? 4 : 2);
        char *dst = reinterpret_cast<char *>(a.out) + samp0 * (IQ16 ? 4 : 2);
        if (NBYTES == 2) *reinterpret_cast<uint16_t *>(dst) = (uint16_t) w[0];
        else if (NBYTES == 4) *reinterpret_cast<uint32_t *>(dst) = w[0];
        else if (NBYTES == 8) *reinterpret_cast<uint2 *>(dst) = make_uint2(w[0], w[1]);
        else {
#pragma unroll
            for (int q = 0; q < NBYTES / 16; q++)
                reinterpret_cast<uint4 *>(dst)[q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
        }
    };

    // One chunk of len (64, or 32 for the tail of a run) consecutive samples.
    auto do_chunk = [&](const int len, int s0) {
        // Chip window of this lane for the chunk (<= 23 chips for 64 samples): 24 chips starting at
        // j0 = (int) code_phase, taken from the periodically extended packed code, XORed with the
        // data bit, and parked at bit 8 so that a right shift by (chip - j0) leaves the
        // "flip the sign" flag where it toggles k by 256: table[k ^ 256] = -table[k].
        const int j0 = __double2loint(__dadd_rz(y, K52));
        const uint32_t lo = ccol[(j0 >> 5) * GROUP], hi = ccol[((j0 >> 5) + 1) * GROUP];
        uint32_t w8 = (__funnelshift_r(lo, hi, j0 & 31) ^ (dbit ? 0xFFFFFFFFu : 0u)) << 8;
        double KY = K52 - (double) j0;
        // table lookup + channel sum of one sample from a VALID (wrapped) NCO state
        auto emit = [&](double xs, double ys) -> int {
            const int k = U32 ? (int) ((u >> 16) & 511u)       // gps.c:2777
                              : __double2loint(__dadd_rz(xs, K43));  // (int) floor(carr_phase*512), gps.c:2775
            const int rel = __double2loint(__dadd_rz(ys, KY)); // (int) code_phase - j0, gps.c:2817
            const int kk = k ^ ((w8 >> rel) & 0x100);          // dataBit*codeCA == -1  <=>  k += 256 (mod 512)
            int e;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(e) : "r"(abase + (uint32_t) kk * 128u));
            return group_sum<GROUP>(e);                        // gps.c:2785-2786 over channels
        };
        // four sums at a time go to the staging row (one 16-byte store; every lane of the group
        // stores the same words)
        auto park = [&](int i, int s0_, int s1_, int s2_, int s3_) {
            *reinterpret_cast<int4 *>(&stage[sub * kChunkMax + i]) = make_int4(s0_, s1_, s2_, s3_);
        };
        // one reference step with its wrap / NAV-bit bookkeeping (gps.c:2789-2826)
        auto step_checked = [&](double &xs, double &ys) {
            if (U32) {
                u += us;                                       // gps.c:2828
                ys = __dadd_rn(ys, dd);
            } else {
                xs = __dadd_rn(xs, cc);
                ys = __dadd_rn(ys, dd);
                if (xs >= 1.0) xs = __dadd_rn(xs, -1.0);       // gps.c:2823-2826
                else if (xs < 0.0) {
                    xs = __dadd_rn(xs, 1.0);
                    if (xs >= 1.0) xs = kBelowOne;            // see nco_exact.h: the phase never reads 1.0
                }
            }
            if (ys >= 1023.0) {                                // gps.c:2791-2813
                ys = __dadd_rn(ys, -1023.0);
                KY = __dadd_rn(KY, 1023.0);                    // the window is periodic in 1023 chips
                if (++icode >= 20) {
                    icode = 0;
                    if (++ibit >= 30) {
                        ibit = 0;
                        ++iword;
                    }
                    const int nb = nav_bit(iword, ibit);
                    if (nb != dbit) w8 = ~w8;
                    dbit = nb;
                }
            }
        };
        // Samples go in groups of 8. A lane can tell in advance whether one of its NCOs can
        // wrap within the next 8 steps (both phases move monotonically inside a block). If no
        // lane of the warp is at risk the group runs with bare additions (the common case,
        // ~3 in 4 groups at 32 channels); otherwise every step carries the reference's wrap /
        // NAV-bit bookkeeping.
        // two groups per loop trip at 32 channels (13.67 -> 13.24 ms); the larger bodies of the 16- and 8-lane
        // variants (shuffle butterflies) do not gain from it
#pragma unroll(GROUP == 32 ? 2 : 1)
        for (int g8 = 0; g8 < len; g8 += 8) {
            const int hx = __double2hiint(x), hy = __double2hiint(y);
            const bool risky = U32 ? hy >= thr_y : (hx >= thr_x_hi) | (hx <= thr_x_lo) | (hy >= thr_y);
            if (!__any_sync(0xFFFFFFFFu, risky)) {
#pragma unroll
                for (int h = 0; h < 8; h += 4) {
                    int sv[4];
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        sv[i] = emit(x, y);
                        if (U32) u += us;                      // gps.c:2828
                        else x = __dadd_rn(x, cc);             // gps.c:2821, no wrap possible
                        y = __dadd_rn(y, dd);                  // gps.c:2789, no wrap possible
                    }
                    park(g8 + h, sv[0], sv[1], sv[2], sv[3]);
                }
            } else {
#pragma unroll
                for (int h = 0; h < 8; h += 4) {
                    int sv[4];
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        sv[i] = emit(x, y);
                        const double xn = U32 ? 0.0 : __dadd_rn(x, cc), yn = __dadd_rn(y, dd);
                        const bool wrap = (!U32 && (unsigned) __double2hiint(xn) >= 0x3FF00000u) |
                                          ((unsigned) __double2hiint(yn) >= 0x408FF800u);
                        if (__any_sync(0xFFFFFFFFu, wrap)) step_checked(x, y);
                        else {
                            if (U32) u += us;
                            else x = xn;
                            y = yn;
                        }
                    }
                    park(g8 + h, sv[0], sv[1], sv[2], sv[3]);
                }
            }
        }
        __syncwarp();
        if (len == 64) flush(std::integral_constant<int, 64>(), s0);
        else flush(std::integral_constant<int, 32>(), s0);
        __syncwarp();
    };

    int s0 = 0;
#pragma unroll 1
    for (; s0 < a.run_samples; s0 += 64)                       // run_samples is a multiple of 32
        do_chunk(a.run_samples - s0 >= 64 ? 64 : 32, s0);
}

// ---------------------------------------------------------------------------------
// Launchers
// ---------------------------------------------------------------------------------
template <int GROUP, bool IQ16, bool U32>
static cudaError_t launch_synth_k(const SynthArgs &a, cudaStream_t s) {
    const int rpw = 32 / GROUP;
    const int warps = (a.runs_per_cta + rpw - 1) / rpw;
    const size_t smem = sizeof(SynthSmem<GROUP>);
    const int ctas = a.nblk * a.ctas_per_block;
    cudaError_t e = cudaFuncSetAttribute(k_synth<GROUP, IQ16, U32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    k_synth<GROUP, IQ16, U32><<<ctas, warps * 32, smem, s>>>(a);
    return cudaGetLastError();
}

template <int GROUP>
static cudaError_t launch_synth_t(const SynthArgs &a, cudaStream_t s) {
    if (a.u32) return a.iq16 ? launch_synth_k<GROUP, true, true>(a, s) : launch_synth_k<GROUP, false, true>(a, s);
    return a.iq16 ? launch_synth_k<GROUP, true, false>(a, s) : launch_synth_k<GROUP, false, false>(a, s);
}

cudaError_t launch_synth(const SynthArgs &a, cudaStream_t s) {
    if (synth_lanes_applicable(a)) return launch_synth_lanes(a, s);
    switch (group_for(a.nchan)) {
        case 32: return launch_synth_t<32>(a, s);
        case 16: return launch_synth_t<16>(a, s);
        default: return launch_synth_t<8>(a, s);
    }
}

void synth_launch_shape(const SynthArgs &a, int *ctas, int *threads, size_t *smem) {
    if (synth_lanes_applicable(a)) return synth_lanes_launch_shape(a, ctas, threads, smem);
    const int grp = group_for(a.nchan), rpw = 32 / grp;
    *ctas = a.nblk * a.ctas_per_block;
    *threads = ((a.runs_per_cta + rpw - 1) / rpw) * 32;
    *smem = grp == 32 ? sizeof(SynthSmem<32>) : (grp == 16 ? sizeof(SynthSmem<16>) : sizeof(SynthSmem<8>));
}

cudaError_t launch_tables(const SynthArgs &a, cudaStream_t s) {
    const long total = (long) a.nblk * 256 * 32;
    k_tables<<<(unsigned) ((total + 255) / 256), 256, 0, s>>>(a, group_for(a.nchan));
    return cudaGetLastError();
}

cudaError_t launch_checkpoints(const SynthArgs &a, cudaStream_t s) {
    const int nblk_pad = (a.nblk + 31) & ~31;
    const long total = (a.u32 ? 1L : 2L) * nblk_pad * a.nchan;      // U32: no carrier walk, code threads only
    const int threads = 128;
    k_checkpoints<<<(unsigned) ((total + threads - 1) / threads), threads, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_probe(const SynthArgs &a, cudaStream_t s) {
    const int nblk_pad = (a.nblk + 31) & ~31;
    const long total = 2L * nblk_pad * a.nchan;
    const int threads = 128;
    k_probe<<<(unsigned) ((total + threads - 1) / threads), threads, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_chain(const SynthArgs &a, cudaStream_t s) {
    const long total = 2L * a.nspan * a.nchan;
    const int threads = 64;
    k_chain<<<(unsigned) ((total + threads - 1) / threads), threads, 0, s>>>(a);
    return cudaGetLastError();
}

}  // namespace gpsb200
