// Core of the LANE = SAMPLE synthesis (k_synth_lanes), shared by the CUDA kernel and by the host model the CPU tests
// compare with the oracle (gpsb200_lanes_model_block).
//
// Idea. The reference advances its two NCOs with one FP64 addition per sample (gps.c:2789-2826). From an EXACT
// state at a run start (RunCkpt, written by k_checkpoints) the true phase after n steps differs from the exact LINEAR
// phase anchor + n * increment only by the accumulated rounding: at most 2^-53 cycles per step for the carrier
// (sums below 2 round to 2^-52, wrap subtraction exact), 2^-44 chips per step for the code (sums below 1024 round
// to 2^-43). So over a run of n <= kMaxRun = 2400 samples (longer runs keep k_synth: the bands below are sized for this)
//     floor(512 * carr_phase) = floor(512 * linear carrier phase)   unless the linear phase lies within
//                               2400 * 2^-53 < 2^-41 cycles of a table-index boundary, and
//     floor(code_phase)       = floor(linear code phase)            unless it lies within 2400 * 2^-44 < 2^-32 chips
//                               of a chip boundary (the code wrap at 1023 chips is one of them).
// The linear phases are kept as 64-bit fixed point (carrier: cycles * 2^64 modulo one cycle; code: chips * 2^54), which
// is exact for every increment the reference can produce above 2^-12 and off by < 2^-64 / 2^-54 per step below. Samples
// whose linear phase falls inside a band are REPAIRED from the exact walk of nco_exact.h; everything else is integer
// arithmetic that a lane can do for ITS sample without knowing its neighbours' -- which is what turns the channel
// dimension into a loop and the sample dimension into lanes.
//
// One window = 96 consecutive samples. Chip signs of a channel for a window are built as three 32-bit words, one per
// residue class r = n mod 3: f_code / f_s = 0.341 chips per sample, so along a residue class the chip index advances
// by 3 * 0.341 = 1 + delta3 (delta3 = 0.023): sample q of the class sits on chip J + q, plus one more after the single
// point where the accumulated q * delta3 carries. A class word is therefore two shifted copies of the chip stream
// spliced at that point.
#pragma once
#include <math.h>
#include <stdint.h>

#include "nco_exact.h"

namespace gpsb200 {
namespace lanes {

constexpr int kWindow = 96;                        // samples per window: 3 residue classes x 32
constexpr int kMaxRun = 2400;                      // longest run the band widths below cover (n * 2^-53 < 2^-41, n * 2^-44 < 2^-32)
constexpr uint64_t kOne54 = 1ull << 54;            // one chip in code fixed point
constexpr uint64_t kCodeWrap54 = 1023ull << 54;    // 1023 chips
constexpr uint64_t kBandCode = 1ull << 22;         // 2^-32 chips
constexpr uint64_t kBandCarr = 1ull << 23;         // 2^-41 cycles (units of 2^-64)
constexpr uint32_t kBandFast = 128;                // units of 2^-32 cycles: slack of the 32-bit per-window phases

// f_code range the residue-class construction needs: 2^-6 <= delta3 = 3 * c_code - 1 < 1/33 (at most one carry per class
// word; the carry point below 64): 1.0157 .. 1.0302 MHz at 3 Msps. GPS L1 C/A is 1.023 MHz +- a few Hz.
GPSB_HD bool code_step_ok(double c_code) { return c_code >= 0.33855 && c_code < 0.34340; }

// carrier phase in [0,1) -> cycles * 2^64 (truncated below 2^-64)
GPSB_HD uint64_t carr_fix(double x) { return (x >= 0.0 && x < 1.0) ? (uint64_t) (x * 0x1p64) : 0; }
// carrier increment in (-1,1) -> two's complement cycles * 2^64
GPSB_HD uint64_t carr_step_fix(double c) {
    const double a = c < 0.0 ? -c : c;
    const uint64_t m = (uint64_t) (a * 0x1p64);
    return c < 0.0 ? (uint64_t) 0 - m : m;
}
GPSB_HD uint64_t code_fix(double y) { return (uint64_t) (y * 0x1p54); }      // chips in [0, 1023) -> chips * 2^54

GPSB_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, int sh) {               // (hi:lo) >> sh, low word, 0 <= sh < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}

// Per (channel, run) state of the lane = channel side.
struct ChanRun {
    uint64_t P, D;          // carrier: linear phase at the current window start, increment per sample
    uint64_t Y, E;          // code: linear phase at the current window start (chips * 2^54, < 1023 * 2^54), increment
    uint32_t inv32;         // floor(2^79 / delta3), delta3 = 3 E - 2^54 in [2^48, 2^49): the carry-point division as a multiply
    uint32_t e22;           // E >> 22: code increment in units of 2^-32 chips (truncated)
    int iword, ibit, icode, dbit;
    bool active;
};

// The exact NCO state at the run start (RunCkpt) and the increments: what the repair paths walk from.
struct Anchor {
    double x0, y0, c, d;
    uint32_t navpos;        // iword | ibit << 8 | icode << 16
};

template <class NavFn>
GPSB_HD int nav_bit_at(NavFn nav, int iw, int ib) {
    const uint32_t w = nav(iw < 60 ? iw : 59);                             // as k_synth: never past the 60-word buffer
    return (int) ((w >> (29 - ib)) & 1u);                                   // gps.c:2812
}

template <class NavFn>
GPSB_HD void init_run(ChanRun &s, bool active, double x, double y, uint32_t navpos, double c, double d, NavFn nav) {
    s.active = active;
    s.iword = (int) (navpos & 0xFF);
    s.ibit = (int) ((navpos >> 8) & 0xFF);
    s.icode = (int) ((navpos >> 16) & 0xFF);
    s.P = carr_fix(x);
    s.D = carr_step_fix(c);
    s.Y = code_fix(y);
    s.E = code_fix(d);
    const uint64_t d3 = 3 * s.E - kOne54;
    s.inv32 = active ? (uint32_t) (0x1p79 / (double) d3) : 0u;                // in (2^30, 2^31]
    s.e22 = (uint32_t) (s.E >> 22);
    s.dbit = active ? nav_bit_at(nav, s.iword, s.ibit) : 0;
}

GPSB_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t) (((uint64_t) a * b) >> 32);
#endif
}

// Second opinion on the carry points of a window, in FP64: used when the 32-bit estimate of window_signs() lands within
// its own error of an integer. c_lo / c_hi: the 64 chip-sign bits from chip j0 on. Returns false when a sample's linear
// code phase is within the band of a chip boundary or a carry point stays ambiguous.
GPSB_HD bool window_signs_fp64(const ChanRun &s, uint32_t c_lo, uint32_t c_hi, int j0, uint32_t S[3]) {
    const uint64_t d3 = 3 * s.E - kOne54;
    const double rinv = 1.0 / (double) d3;
    const double tband = (double) kBandCode * rinv + 0x1p-40;                // band of the carry-point test, in units of q
    bool certain = true;
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const uint64_t phi = s.Y + (uint64_t) r * s.E;
        const int J = (int) (phi >> 54) - j0;                                 // 0 or 1
        const uint64_t F = phi & (kOne54 - 1);
        // carry point: smallest q with F + q * d3 >= 1 chip. FP64 is exact enough OUTSIDE the band tested below:
        // (1 - F) / d3 is at most 2^-45 off, the band is >= 2^-40.
        const double t = (double) (kOne54 - F) * rinv;
        const double tf = t < 64.0 ? (double) (int) t : 64.0;                 // floor (t > 0)
        const int qs = (int) tf + 1;
        certain &= F >= kBandCode;
        if (qs <= 32) certain &= (t - tf >= tband) & (tf + 1.0 - t >= tband);
        const uint32_t lowm = qs >= 32 ? 0xFFFFFFFFu : ((1u << qs) - 1u);
        const uint32_t a = funnel_r(c_lo, c_hi, J), b = funnel_r(c_lo, c_hi, J + 1);
        S[r] = (a & lowm) | (b & ~lowm);
    }
    return certain;
}

// The chip-sign words of the current window: S[r] bit q = sign flag (chip XOR data bit) of sample 3q + r.
// chips(w) = word w of the channel's packed, periodically extended C/A code (bit n = ca[n mod 1023]).
// Returns false when some sample's linear code phase is too close to a chip boundary (or the carry point of a class is
// ambiguous): the caller then builds the words with exact_signs().
// 32-bit integer arithmetic only on the common path. Code phases are taken in units of 2^-32 chips (f0 = Y >> 22, e22 =
// E >> 22): the fraction of class r, fr = f0 + r e22 (mod one chip), is short of the true one by at most 2 units, so the
// chip offset J (its carry) is certain when fr keeps 4 units away from the wrap -- which also covers the band condition
// of sample 0 (2^-32 chips = 1 unit). The carry point t = (1 chip - F) / delta3 is estimated from below as
// mulhi32(2^32 - fr - 3, inv32) = t * 2^25, short by less than 2^-22 (truncations of fr, inv32 and the product); when its
// fraction keeps 2^-21 away from 0 and 1 the floor is certain and so is the band condition of the carry point (<= 2^-26).
template <class ChipFn, class NavFn>
GPSB_HD bool window_signs(const ChanRun &s, ChipFn chips, NavFn nav, uint32_t S[3], bool force_fp64 = false) {
    const int j0 = (int) (s.Y >> 54);
    // 64 chips from chip j0 on, data bit folded in; chips of the NEXT code period (position >= 1023 - j0) take the
    // next NAV bit when this period is the 20th of its bit (gps.c:2793-2812)
    const int wi = j0 >> 5, sh = j0 & 31;
    const uint32_t w0 = chips(wi), w1 = chips(wi + 1), w2 = chips(wi + 2);
    uint32_t c_lo = funnel_r(w0, w1, sh), c_hi = funnel_r(w1, w2, sh);
    if (s.dbit) {
        c_lo = ~c_lo;
        c_hi = ~c_hi;
    }
    const int pw = 1023 - j0;
    if (pw < 64 && s.icode == 19) {
        int ib = s.ibit + 1, iw = s.iword;
        if (ib >= 30) {
            ib = 0;
            ++iw;
        }
        if (nav_bit_at(nav, iw, ib) != s.dbit) {
            if (pw < 32) {
                c_lo ^= 0xFFFFFFFFu << pw;
                c_hi = ~c_hi;
            } else {
                c_hi ^= 0xFFFFFFFFu << (pw - 32);
            }
        }
    }
    const uint32_t f0 = (uint32_t) (s.Y >> 22);
    const uint32_t sh1 = funnel_r(c_lo, c_hi, 1), sh2 = funnel_r(c_lo, c_hi, 2);
    bool certain = !force_fp64;
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const uint32_t fr = f0 + (uint32_t) r * s.e22;                        // r e22 < one chip: at most one wrap
        const bool J = fr < f0;                                               // chip offset of the class: 0 or 1
        certain &= fr + 4u >= 8u;                                             // 4 <= fr < 2^32 - 4
        const uint32_t t25 = mulhi32(~fr - 2u, s.inv32);
        const uint32_t fl = t25 >> 25, frac = t25 & ((1u << 25) - 1u);
        certain &= (fl >= 32u) | ((frac >= 16u) & (frac < (1u << 25) - 16u));
        const uint32_t lowm = fl >= 31u ? 0xFFFFFFFFu : ((2u << fl) - 1u);    // samples q < fl + 1 precede the carry
        const uint32_t a = J ? sh1 : c_lo, b = J ? sh2 : sh1;
        S[r] = (a & lowm) | (b & ~lowm);
    }
    if (certain) return true;
    return window_signs_fp64(s, c_lo, c_hi, j0, S);
}

// Next window: 96 samples on.
template <class NavFn>
GPSB_HD void advance_window(ChanRun &s, NavFn nav) {
    s.P += (uint64_t) kWindow * s.D;
    const uint64_t y_old = s.Y;
    s.Y += (uint64_t) kWindow * s.E;                                          // 1023 + 33 chips passes 2^64: modular
    if (s.Y < y_old || s.Y >= kCodeWrap54) {
        s.Y -= kCodeWrap54;
        if (++s.icode >= 20) {
            s.icode = 0;
            if (++s.ibit >= 30) {
                s.ibit = 0;
                ++s.iword;
            }
            s.dbit = nav_bit_at(nav, s.iword, s.ibit);
        }
    }
}

// Exact chip-sign words of window w of the run (repair path): the reference's own code recurrence, stepped sample by
// sample from the exact state at the window start (nco_exact.h).
template <class ChipFn, class NavFn>
GPSB_HD void exact_signs(const Anchor &an, int w, ChipFn chips, NavFn nav, uint32_t S[3]) {
    double y = an.y0;
    int iword = (int) (an.navpos & 0xFF), ibit = (int) ((an.navpos >> 8) & 0xFF), icode = (int) ((an.navpos >> 16) & 0xFF);
    int64_t periods = 0;
    nco_advance<NCO_CODE>(y, an.d, (int64_t) w * kWindow, periods);
    nav_advance(iword, ibit, icode, periods);
    int dbit = nav_bit_at(nav, iword, ibit);
    S[0] = S[1] = S[2] = 0;
    for (int n = 0; n < kWindow; n++) {
        const int j = (int) y;                                              // gps.c:2817
        const uint32_t chip = (chips(j >> 5) >> (j & 31)) & 1u;
        const uint32_t flag = chip ^ (uint32_t) dbit;
        const int q = n / 3, r = n - 3 * q;
        S[r] |= flag << q;
        int64_t p = 0;
        nco_step<NCO_CODE>(y, an.d, p);
        if (p) {
            if (++icode >= 20) {
                icode = 0;
                if (++ibit >= 30) {
                    ibit = 0;
                    ++iword;
                }
                dbit = nav_bit_at(nav, iword, ibit);
            }
        }
    }
}

// Carrier table index of sample n of a window whose linear start phase is P (increment D), certain by construction:
// 64-bit linear phase, and the exact walk from the run anchor when that lies inside the band (w = window number within
// the run).
GPSB_HD int exact_index(uint64_t P, uint64_t D, const Anchor &an, int w, int n, bool force_walk = false) {
    const uint64_t m = P + (uint64_t) n * D;
    const uint64_t frac = m & ((1ull << 55) - 1);
    if (!force_walk && frac >= kBandCarr && frac <= (1ull << 55) - kBandCarr) return (int) (m >> 55);
    double x = an.x0;
    int64_t dummy = 0;
    nco_advance<NCO_CARRIER>(x, an.c, (int64_t) w * kWindow + n, dummy);
#if defined(__CUDA_ARCH__)
    return __double2loint(__dadd_rz(x, 8796093022208.0)) & 511;              // (int) floor(x * 512), gps.c:2775
#else
    return (int) (x * 512.0) & 511;
#endif
}

// What the lane = sample side works from in a window: 32-bit phase of sample 0 (biased by -1 so that the true phase is
// strictly above it) and the increment per sample, both truncated: sample n's true 32-bit phase lies in
// (base + n * d1, base + n * d1 + 98), so the index taken from base + n * d1 is right unless its fraction is within
// kBandFast of the next boundary -- fast_risky().
// Integer carrier NCO of the reference (GPSB200_CARRIER_U32): carr_phasestep = (int) round(512.0 * 65536.0 * f_carr * delt),
// gps.c:2746 -- left to right with the constant product folded (two roundings, no FMA), C round (ties away from zero).
// Host only: the kernels read it from BlockChanDev::step_u32.
inline int32_t u32_carrier_step(double f_carr) { return (int32_t) round((33554432.0 * f_carr) * (1.0 / 3000000.0)); }

GPSB_HD uint32_t fast_base(const ChanRun &s) { return (uint32_t) (s.P >> 32) - 1u; }
GPSB_HD uint32_t fast_step(const ChanRun &s) { return (uint32_t) (s.D >> 32); }
GPSB_HD bool fast_risky(uint32_t p) { return (((~p) << 9) < (kBandFast << 9)); }

}  // namespace lanes
}  // namespace gpsb200
