// k_synth_lanes: the per-sample synthesis (gps.c:2767-2857) with LANE = SAMPLE.
//
// k_synth (synth_kernels.cu) puts the channels on the lanes and pays a warp reduction per sample (and FP64 additions for
// both NCOs of every channel-sample); with 12 channels a quarter of its lanes idle and the reduction is a shuffle
// butterfly. Here a lane owns three samples of a 96-sample window and loops over the channels of the call, accumulating
// in registers: integer work only, proportional to the channel count.
// What makes that possible is synth_lanes.h: from the exact run anchors of k_checkpoints both NCO phases of any sample are
// integer arithmetic on certified fixed-point linear phases; the rare samples a band test cannot certify are repaired
// from the exact FP64 walk of nco_exact.h. The algorithm is the one the host model (lanes_model.cpp) runs against the
// oracle in the CPU tests; this file only distributes it over a warp:
//
//   channel side  up to 16 channels: lane = (half h, channel c), state of channel c at window w + h of the warp's run,
//                 every trip produces the chip-sign words and the 32-bit phase base of TWO windows into shared memory;
//                 17..32 channels: lane = channel, one window per trip
//   sample side   lane q: samples 3q, 3q+1, 3q+2 of each window of the trip: per channel one broadcast read of the
//                 window record, three table look-ups (index and sign from one 32-bit word), register accumulation
//   output        quantise + pack (gps.c:2833-2845), staged per warp, written with 16-byte stores
#include <cuda_runtime.h>
#include <stdint.h>

#include "nco_exact.h"
#include "synth_kernels.h"
#include "synth_lanes.h"

namespace gpsb200 {

namespace {

constexpr int kLaneWarps = 16;
constexpr int kLaneChipWords = 36;      // 1023 chips periodically extended to 1152 bits (window_signs reads word j0/32 + 2)

struct LaneWin {
    uint32_t s0, s1, s2;                // chip-sign words of the residue classes (bit q: sample 3q + r)
    uint32_t base;                      // 32-bit carrier phase of sample 0, biased by -1 (fast_base)
};

// CH = channel capacity of the variant (16 or 32). The channel side uses all 32 lanes: with CH = 16 the two half-warps
// prepare two consecutive windows per trip, with CH = 32 the warp prepares one.
// The carrier tables ([channel][k]: I + (Q << 16), gain-scaled, gps.c:2781-2782; 2 KB per channel) sit in front of this
// struct at a 2 KB-aligned shared address, so that "table base | byte offset of k" is one logic instruction. Entry k of
// channel c is stored at k ^ swz(c) (swz(c) = c * 32 / CH): the transposing fill from k_tables' [k][channel] layout is then
// free of bank conflicts, and the look-ups fold the swizzle into the same logic instruction ("^ (base | swz)").
template <int CH>
struct LanesSmem {
    static constexpr int kWins = 32 / CH;
    uint32_t chips[CH][kLaneChipWords];                 // packed C/A chips, bit n = ca[n mod 1023]
    uint32_t nav[CH][kNavWords];                        // NAV words of this block's frame
    alignas(16) LaneWin win[kLaneWarps][kWins][CH];     // per warp: the window(s) in flight
    alignas(16) uint32_t step[kLaneWarps][CH];          // per warp: 32-bit carrier increment per sample (fast_step)
    alignas(16) uint32_t stage[kLaneWarps][kWins * lanes::kWindow];   // packed output of the window(s)
};
template <int CH>
constexpr size_t lanes_smem_bytes() { return sizeof(LanesSmem<CH>) + (size_t) CH * 2048 + 2048; }

__device__ __forceinline__ uint64_t shfl64(uint64_t v, int src) {
    const uint32_t lo = __shfl_sync(0xFFFFFFFFu, (uint32_t) v, src);
    const uint32_t hi = __shfl_sync(0xFFFFFFFFu, (uint32_t) (v >> 32), src);
    return ((uint64_t) hi << 32) | lo;
}

// U32: the reference's integer carrier build (gps.c:2777, 2828). Sample n of a run has the EXACT phase u_run + n * step
// (mod 2^32), so the window record carries (u_run + 96 w step) << 7 and the sample side adds n * (step << 7): the index
// (u >> 16) & 511 lands in bits 23..31 as in the FP64 variant, and the chip sign folds in as bit 31 the same way. What
// only the FP64 carrier needs is compiled out: the 64-bit linear phase (ChanRun::P/D is then dead), the band tracking
// (VIMNMX3), the per-window vote and the repair.
template <bool IQ16, int CH, bool U32>
__global__ void __launch_bounds__(kLaneWarps * 32, 2) k_synth_lanes(SynthArgs a) {
    constexpr int WINS = 32 / CH;                     // windows per trip
    constexpr int SWZ = 32 / CH;                      // swz(c) = c * SWZ
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t raw_base = (uint32_t) __cvta_generic_to_shared(smem_raw);
    const uint32_t tab_base = (raw_base + 2047u) & ~2047u;
    int32_t *tab = reinterpret_cast<int32_t *>(smem_raw + (tab_base - raw_base));                 // [channel][512]
    LanesSmem<CH> &sm = *reinterpret_cast<LanesSmem<CH> *>(smem_raw + (tab_base - raw_base) + CH * 2048);
    constexpr uint32_t kFull = 0xFFFFFFFFu;

    const int b = blockIdx.x / a.ctas_per_block;
    const int g = blockIdx.x - b * a.ctas_per_block;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int nchan = a.nchan;
    const BlockChanDev *bc = a.bc + (size_t) b * nchan;

    // ---- per-CTA tables ----------------------------------------------------------------------------------
    {
        const int32_t *src = a.atab + (size_t) b * kAtabRows * 32;             // [k][lane], column c = channel c
        for (int i = tid; i < 512 * CH; i += nthr) {
            const int k = i / CH, c = i - k * CH;
            tab[c * 512 + (k ^ (c * SWZ))] = c < nchan ? src[k * 32 + c] : 0;
        }
        for (int i = tid; i < CH * kLaneChipWords; i += nthr) {
            const int c = i / kLaneChipWords, w = i - c * kLaneChipWords;
            uint32_t v = 0;
            if (c < nchan && bc[c].prn > 0) {
                const uint32_t *cw = a.chipbits + bc[c].prn * kChipWords;        // 33 words: bits 0 .. 1055
                // bit n of the extension = bit n - 1023 = bit 32 (w - 32) + i + 1 of the stream
                v = w < kChipWords ? cw[w] : __funnelshift_r(cw[w - 32], cw[w - 31], 1);
            }
            sm.chips[c][w] = v;
        }
        for (int i = tid; i < CH * kNavWords; i += nthr) {
            const int c = i / kNavWords, w = i - c * kNavWords;
            uint32_t v = 0;
            if (c < nchan && bc[c].prn > 0) v = a.nav[((size_t) bc[c].frame * a.nav_stride + c) * kNavWords + w];
            sm.nav[c][w] = v;
        }
    }
    __syncthreads();

    // ---- roles of this lane -----------------------------------------------------------------------------------
    const int ch = lane & (CH - 1), half = lane / CH;                            // channel side
    const bool chan_ok = ch < nchan && bc[ch < nchan ? ch : 0].prn > 0;
    const uint32_t *nav_row = &sm.nav[ch][0];
    const uint32_t *chip_row = &sm.chips[ch][0];
    auto navf = [nav_row](int iw) { return nav_row[iw]; };
    auto chipf = [chip_row](int i) { return chip_row[i]; };
    const uint32_t lane3 = 3u * (uint32_t) lane;                                  // sample side
    uint32_t pw;                             // bit lane -> bit 31 by a MULTIPLICATION (FMA pipe): opaque to the compiler,
    asm volatile("mov.b32 %0, %1;" : "=r"(pw) : "r"(1u << (31 - lane)));          // which would turn it back into a shift
    const int nwin = a.run_samples / lanes::kWindow;
    uint32_t *stage = &sm.stage[warp][0];

    const int run_first = g * a.runs_per_cta;
    const int run_last = min(run_first + a.runs_per_cta, a.nruns);
#pragma unroll 1
    for (int r = run_first + warp; r < run_last; r += kLaneWarps) {
        // ---- channel side: exact anchor of (run, channel), window state of window 0 + half -------------------------
        lanes::ChanRun s;
        lanes::Anchor an = {0.0, 0.0, 0.0, 0.0, 0u};
        if (chan_ok) {
            const RunCkpt k0 = a.ck[((size_t) b * a.nruns + r) * nchan + ch];
            an.x0 = k0.x;
            an.y0 = k0.y;
            an.navpos = k0.nav;
            an.c = bc[ch].c_carr;
            an.d = bc[ch].c_code;
        }
        lanes::init_run(s, chan_ok, an.x0, an.y0, an.navpos, an.c, an.d, navf);
        if (!chan_ok) s.P = s.D = s.Y = s.E = 0;
        // U32 carrier of this lane's channel: phase << 7 at the current window start, step << 7
        const uint32_t ust = U32 && chan_ok ? (uint32_t) bc[ch].step_u32 << 7 : 0u;
        uint32_t ub = U32 && chan_ok ? (uint32_t) an.x0 << 7 : 0u;
        if (half == 0) sm.step[warp][ch] = chan_ok ? (U32 ? ust : lanes::fast_step(s)) : 0u;
        if (WINS == 2 && chan_ok && half == 1) {
            lanes::advance_window(s, navf);
            ub += (uint32_t) lanes::kWindow * ust;
        }
        const size_t samp0 = (size_t) b * kBlockSamples + (size_t) r * a.run_samples;

#pragma unroll 1
        for (int w = 0; w < nwin; w += WINS) {
            {
                uint32_t S[3] = {0u, 0u, 0u};
                uint32_t base = 0u;
                if (chan_ok && w + half < nwin) {
                    if (!lanes::window_signs(s, chipf, navf, S)) lanes::exact_signs(an, w + half, chipf, navf, S);
                    base = U32 ? ub : lanes::fast_base(s);
                }
                *reinterpret_cast<uint4 *>(&sm.win[warp][half][ch]) = make_uint4(S[0], S[1], S[2], base);
            }
            __syncwarp();

            // ---- sample side ------------------------------------------------------------------------------------
#pragma unroll
            for (int hh = 0; hh < WINS; hh++) {
                if (w + hh >= nwin) break;
                const LaneWin *wrow = &sm.win[warp][hh][0];
                int acc0 = 0, acc1 = 0, acc2 = 0;
                uint32_t dmax = 0u;
                // Two channels per trip (an odd count is padded with the next slot, which is all zeros). The integer work is
                // split over both integer pipes on purpose (ncu: the ALU pipe was the limiter at 81 % with the FMA pipe at 21 %):
                // the sign bit reaches bit 31 through a multiplication by the lane's power of two.
#pragma unroll 4
                for (int c = 0; c < nchan; c += 2) {
                    const uint4 wa = *reinterpret_cast<const uint4 *>(&wrow[c]);      // broadcast
                    const uint4 wb = *reinterpret_cast<const uint4 *>(&wrow[c + 1]);
                    const uint2 st = *reinterpret_cast<const uint2 *>(&sm.step[warp][c]);
                    const uint32_t a0 = wa.w + lane3 * st.x, a1 = a0 + st.x, a2 = a1 + st.x;
                    const uint32_t b0 = wb.w + lane3 * st.y, b1 = b0 + st.y, b2 = b1 + st.y;
                    // chip x data-bit sign = half a cycle: table[k ^ 256] = -table[k]
                    const uint32_t qa0 = a0 ^ ((wa.x * pw) & 0x80000000u), qa1 = a1 ^ ((wa.y * pw) & 0x80000000u),
                                   qa2 = a2 ^ ((wa.z * pw) & 0x80000000u);
                    const uint32_t qb0 = b0 ^ ((wb.x * pw) & 0x80000000u), qb1 = b1 ^ ((wb.y * pw) & 0x80000000u),
                                   qb2 = b2 ^ ((wb.z * pw) & 0x80000000u);
                    // table base (low 11 bits zero) | swizzle of the channel as a byte offset (< 128): linear in c
                    const uint32_t ta = tab_base + (uint32_t) c * (2048u + 4u * SWZ), tb = ta + (2048u + 4u * SWZ);
                    int ea0, ea1, ea2, eb0, eb1, eb2;
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(ea0) : "r"(((qa0 >> 21) & 0x7FCu) ^ ta));
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(eb0) : "r"(((qb0 >> 21) & 0x7FCu) ^ tb));
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(ea1) : "r"(((qa1 >> 21) & 0x7FCu) ^ ta));
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(eb1) : "r"(((qb1 >> 21) & 0x7FCu) ^ tb));
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(ea2) : "r"(((qa2 >> 21) & 0x7FCu) ^ ta));
                    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(eb2) : "r"(((qb2 >> 21) & 0x7FCu) ^ tb));
                    acc0 += ea0 + eb0;
                    acc1 += ea1 + eb1;
                    acc2 += ea2 + eb2;
                    // fast_risky(p) <=> (~p) << 9 < kBandFast << 9 <=> p << 9 > 0xFFFFFE00 - (kBandFast << 9): the largest
                    // fraction below an index boundary over all channels and samples (the sign bit shifts out)
                    if (!U32) {
                        dmax = __vimax3_u32(dmax, qa0 << 9, qb0 << 9);
                        dmax = __vimax3_u32(dmax, qa1 << 9, qb1 << 9);
                        dmax = __vimax3_u32(dmax, qa2 << 9, qb2 << 9);
                    }
                }
                if (!U32 && __any_sync(kFull, dmax > 0xFFFFFE00u - (lanes::kBandFast << 9))) {
                    // ---- repair: some sample of this window sits within 2^-25 cycles below an index boundary for some
                    // channel. Find the channel(s), take the certain index of exactly those (channel, sample) pairs (64-bit
                    // linear phase; exact walk from the run anchor inside the 2^-41 band) and patch the sums.
                    for (int c = 0; c < nchan; c++) {
                        const uint4 wv = *reinterpret_cast<const uint4 *>(&wrow[c]);
                        const uint32_t st = sm.step[warp][c];
                        const uint32_t p0 = wv.w + lane3 * st, p1 = p0 + st, p2 = p1 + st;
                        const bool risky = lanes::fast_risky(p0) | lanes::fast_risky(p1) | lanes::fast_risky(p2);
                        if (!__any_sync(kFull, risky)) continue;
                        const int src = hh * CH + c;
                        const uint64_t Pc = shfl64(s.P, src), Dc = shfl64(s.D, src);
                        if (!risky || bc[c].prn <= 0) continue;
                        const RunCkpt k0 = a.ck[((size_t) b * a.nruns + r) * nchan + c];
                        const lanes::Anchor ac = {k0.x, k0.y, bc[c].c_carr, bc[c].c_code, k0.nav};
                        const uint32_t ps[3] = {p0, p1, p2}, sw[3] = {wv.x, wv.y, wv.z};
                        int fix[3] = {0, 0, 0};
#pragma unroll
                        for (int rr = 0; rr < 3; rr++) {
                            if (!lanes::fast_risky(ps[rr])) continue;
                            const int kf = (int) (ps[rr] >> 23);
                            const int k = lanes::exact_index(Pc, Dc, ac, w + hh, (int) lane3 + rr);
                            const int flip = (int) ((sw[rr] >> lane) & 1u) << 8;
                            fix[rr] = tab[c * 512 + ((k ^ flip) ^ (c * SWZ))] - tab[c * 512 + ((kf ^ flip) ^ (c * SWZ))];
                        }
                        acc0 += fix[0];
                        acc1 += fix[1];
                        acc2 += fix[2];
                    }
                }
                // ---- quantise + pack (gps.c:2833-2845) ---------------------------------------------------------------
                const int accs[3] = {acc0, acc1, acc2};
#pragma unroll
                for (int rr = 0; rr < 3; rr++) {
                    const int p = accs[rr];
                    const int iv = (int) (short) (p & 0xFFFF);                 // (short) i_acc, gps.c:2834
                    const int qv = (p - iv) >> 16;                             // (short) q_acc, gps.c:2835
                    const int n = hh * lanes::kWindow + (int) lane3 + rr;
                    if (IQ16) {
                        stage[n] = ((uint32_t) iv & 0xFFFFu) | ((uint32_t) qv << 16);
                    } else {
                        reinterpret_cast<uint16_t *>(stage)[n] =
                            (uint16_t) ((((uint32_t) (iv >> 4)) & 0xFFu) | ((((uint32_t) (qv >> 4)) & 0xFFu) << 8));  // gps.c:2844
                    }
                }
            }
            __syncwarp();
            // ---- 16-byte stores of the window(s) of this trip ------------------------------------------------------------
            {
                const int nsamp = (nwin - w >= WINS ? WINS : 1) * lanes::kWindow;
                const int nvec = nsamp * (IQ16 ? 4 : 2) / 16;
                uint4 *dst = reinterpret_cast<uint4 *>(reinterpret_cast<char *>(a.out) +
                                                       (samp0 + (size_t) w * lanes::kWindow) * (IQ16 ? 4 : 2));
                const uint4 *srcv = reinterpret_cast<const uint4 *>(stage);
                for (int i = lane; i < nvec; i += 32) dst[i] = srcv[i];
            }
            if (chan_ok) {
#pragma unroll
                for (int i = 0; i < WINS; i++) lanes::advance_window(s, navf);
                ub += (uint32_t) (WINS * lanes::kWindow) * ust;
            }
        }
    }
}

}  // namespace

bool synth_lanes_applicable(const SynthArgs &a) {
    return a.lanes && a.nchan <= 32 && a.run_samples % lanes::kWindow == 0 && a.run_samples <= lanes::kMaxRun &&
           (reinterpret_cast<uintptr_t>(a.out) & 15u) == 0;                    // 16-byte stores
}

static void lanes_shape(const SynthArgs &a, int *ctas_per_block, int *runs_per_cta) {
    // CTAs all take about the same time and 2 x 148 of them are resident: aim at 40 or more waves so that the last,
    // partly filled one costs little (2999 blocks as ONE CTA each are 10.1 waves -> 11: 8 % lost), in steps of one run
    // per warp of a CTA
    int per_block = (40 * 2 * 148 + a.nblk - 1) / a.nblk;
    if (per_block > 16) per_block = 16;
    if (per_block < 1) per_block = 1;
    int per_cta = (a.nruns + per_block - 1) / per_block;
    per_cta = (per_cta + kLaneWarps - 1) / kLaneWarps * kLaneWarps;
    per_block = (a.nruns + per_cta - 1) / per_cta;
    *ctas_per_block = per_block;
    *runs_per_cta = per_cta;
}

template <bool IQ16, int CH, bool U32>
static cudaError_t launch_lanes_t(const SynthArgs &a, cudaStream_t s) {
    const size_t smem = lanes_smem_bytes<CH>();
    cudaError_t e = cudaFuncSetAttribute(k_synth_lanes<IQ16, CH, U32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    k_synth_lanes<IQ16, CH, U32><<<a.nblk * a.ctas_per_block, kLaneWarps * 32, smem, s>>>(a);
    return cudaGetLastError();
}

template <bool U32>
static cudaError_t launch_lanes_mode(const SynthArgs &a, cudaStream_t s) {
    if (a.nchan <= 16) return a.iq16 ? launch_lanes_t<true, 16, U32>(a, s) : launch_lanes_t<false, 16, U32>(a, s);
    return a.iq16 ? launch_lanes_t<true, 32, U32>(a, s) : launch_lanes_t<false, 32, U32>(a, s);
}

cudaError_t launch_synth_lanes(const SynthArgs &a_in, cudaStream_t s) {
    SynthArgs a = a_in;
    lanes_shape(a, &a.ctas_per_block, &a.runs_per_cta);
    return a.u32 ? launch_lanes_mode<true>(a, s) : launch_lanes_mode<false>(a, s);
}

void synth_lanes_launch_shape(const SynthArgs &a, int *ctas, int *threads, size_t *smem) {
    int per_block, per_cta;
    lanes_shape(a, &per_block, &per_cta);
    *ctas = a.nblk * per_block;
    *threads = kLaneWarps * 32;
    *smem = a.nchan <= 16 ? lanes_smem_bytes<16>() : lanes_smem_bytes<32>();
}

}  // namespace gpsb200
