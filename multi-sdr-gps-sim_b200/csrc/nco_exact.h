// Exact fast-forward of the reference's double-precision NCO recurrences.
//
// The reference advances two phases once per sample, in IEEE binary64 with a
// separately rounded add (no FMA; -std=c11 => -ffp-contract=off):
//   code   : x += c; if (x >= 1023.0) { x -= 1023.0; ++periods; }      (gps.c:2789-2793)
//   carrier: x += c; if (x >= 1.0) x -= 1.0; else if (x < 0.0) x += 1.0; (gps.c:2821-2826)
// with c = fl(f * delt) constant inside a 0.1 s block. Bit-exact output needs the
// exact x after n steps, not x0 + n*c (SURVEY.md hard part 1).
//
// Observation used here: while x stays inside one binade [2^e, 2^(e+1)) and does not
// wrap, x = X*u (u = 2^(e-52), X a 53-bit integer) and fl(x + c) = (X + R)*u with a
// CONSTANT integer R = round-to-nearest(c/u) (on an exact tie: the even one of the two
// neighbours, once X is even). So a run of k in-binade steps is X += k*R, and only the
// steps that cross a binade boundary or wrap are executed as real additions.
// nco_advance() therefore costs O(#binade crossings) instead of O(n).
//
// Shared by host code (carrier-phase chain across blocks) and device code (run
// checkpoints), hence the GPSB_HD qualifier and the absence of libm calls.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define GPSB_HD __host__ __device__ __forceinline__
#else
#define GPSB_HD inline
#endif

namespace gpsb200 {

enum NcoKind { NCO_CODE = 0, NCO_CARRIER = 1 };

// Largest double below 1.0. The reference's negative-Doppler wrap `carr_phase += 1.0`
// (gps.c:2825-2826) can round a tiny negative phase to exactly 1.0, after which its table
// index (int) floor(1.0 * 512) = 512 reads past cosTable512/sinTable512 (gps.c:2775-2782):
// undefined behaviour, probability ~2^-54/|c| per wrap. This implementation (and the test
// oracle) clamp that one value to 1 - 2^-53 instead, which keeps the index at 511.
constexpr double kBelowOne = 0.99999999999999988897769753748434595763683319091796875;

GPSB_HD uint64_t f64_bits(double v) {
#if defined(__CUDA_ARCH__)
    return (uint64_t) __double_as_longlong(v);
#else
    uint64_t b;
    memcpy(&b, &v, 8);
    return b;
#endif
}

GPSB_HD double bits_f64(uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long) b);
#else
    double v;
    memcpy(&v, &b, 8);
    return v;
#endif
}

// A k with k <= floor(room / d), never more than one short of it (room, d < 2^53).
// Any such k is valid for the jump; only the iteration count depends on it. The device
// version avoids the (slow, ~100-instruction) 64-bit integer division.
GPSB_HD uint64_t safe_quotient(uint64_t room, uint64_t d) {
#if defined(__CUDA_ARCH__)
    // both operands convert exactly; rcp and mul each err by <= 2^-53 relative; shaving
    // 2^-49 guarantees q <= room/d.
    const double q = __dmul_rd(__dmul_rd((double) room, __drcp_rd((double) d)), 1.0 - 0x1p-49);
    return (uint64_t) __double2ull_rd(q);
#else
    return room / d;
#endif
}

// One step exactly as the reference performs it. `periods` counts code wraps.
template <int KIND>
GPSB_HD void nco_step(double &x, double c, int64_t &periods) {
#if defined(__CUDA_ARCH__)
    x = __dadd_rn(x, c);
#else
    x = x + c;
#endif
    if (KIND == NCO_CODE) {
        if (x >= 1023.0) {
            x -= 1023.0;
            ++periods;
        }
    } else {
        if (x >= 1.0) x -= 1.0;
        else if (x < 0.0) {
            x += 1.0;
            if (x >= 1.0) x = kBelowOne;
        }
    }
}

// Advance x by exactly n reference steps of increment c -- integer-lattice formulation
// (any c; used for degenerate increments and as the cross-check of the fast version below).
// Returns the number of loop iterations spent (diagnostics only).
template <int KIND>
GPSB_HD int nco_advance_generic(double &x, double c, int64_t n, int64_t &periods) {
    const uint64_t MANT = (1ull << 52) - 1;
    int iters = 0;
    if (c == 0.0 || n <= 0) return 0;
    const bool neg = c < 0.0;
    const uint64_t cb = f64_bits(c) & 0x7FFFFFFFFFFFFFFFull;   // |c|
    const int ec = (int) (cb >> 52);
    const uint64_t cm = (cb & MANT) | (1ull << 52);
    const double ac = bits_f64(cb);
    // Mantissa-domain upper bound of the wrap threshold in its own binade:
    // 1023.0 = 0x3FF<<... lives in binade [512,1024): 1023 * 2^43; 1.0 is a binade edge.
    const int e_wrap = (KIND == NCO_CODE) ? (1023 + 9) : -1;
    const uint64_t x_wrap = 1023ull << 43;

    while (n > 0) {
        ++iters;
        const uint64_t xb = f64_bits(x);
        const int ex = (int) ((xb >> 52) & 0x7FF);
        // Below |c| (incl. zero, negatives, subnormals), or c subnormal: plain step.
        if ((xb >> 63) || !(x >= ac) || ec == 0) {
            nco_step<KIND>(x, c, periods);
            --n;
            continue;
        }
        const int sh = ex - ec;                  // >= 0 because x >= |c|
        if (sh >= 54) return iters;              // |c| < ulp(x)/2: x + c == x for ever
        uint64_t X = (xb & MANT) | (1ull << 52);
        uint64_t Cq = cm >> sh;
        uint64_t R = Cq;
        if (sh > 0) {
            const uint64_t rem = cm & ((1ull << sh) - 1);
            const uint64_t half = 1ull << (sh - 1);
            if (rem > half) R = Cq + 1;
            else if (rem == half) {              // exact tie: result mantissa is even
                if (X & 1) {                     // one real step makes X even
                    nco_step<KIND>(x, c, periods);
                    --n;
                    continue;
                }
                R = (Cq & 1) ? Cq + 1 : Cq;
            }
        }
        if (R == 0) return iters;                // increment rounds away: fixed point
        // Steps that provably stay strictly inside the binade (and below the wrap
        // threshold); Cq+1 >= R keeps every intermediate REAL sum inside as well.
        uint64_t room;
        if (!neg) {
            uint64_t hi = (KIND == NCO_CODE && ex == e_wrap) ? x_wrap : (1ull << 53);
            room = hi - 1 - X;
        } else {
            room = X - (1ull << 52);
        }
        uint64_t k = safe_quotient(room, Cq + 1);
        if (k > (uint64_t) n) k = (uint64_t) n;
        if (k > 0) {
            X = neg ? X - k * R : X + k * R;
            x = bits_f64(((uint64_t) ex << 52) | (X & MANT));
            n -= (int64_t) k;
        }
        if (n > 0) {                             // boundary / wrap (or filler) step, done for real
            nco_step<KIND>(x, c, periods);
            --n;
        }
    }
    return iters;
}

// ---------------------------------------------------------------------------------
// Fast formulation of the same walk: all lattice quantities come out of FP64 itself.
//   * the in-binade step R*u is c rounded to the binade's grid: (2^e + |c|) - 2^e
//     (round-half-even there == "the even neighbour" on an exact tie);
//   * the number of steps that provably stay inside is floor(room * rinv), rinv a
//     slightly shrunk 1/|c| (valid while ulp(x)/|c| <= 2^-30, i.e. |c| >= 2^-23);
//   * k * (R*u) and x + k*(R*u) are exact in double (k*R < 2^53).
// Every iteration executes the same instruction sequence (selects, no data-dependent
// branches besides the loop itself), which keeps the lanes of a GPU warp together.
struct WalkConst {
    double c, ac, rinv;
    int ec;
    bool neg, fast;
};

GPSB_HD WalkConst walk_const(double c) {
    WalkConst w;
    w.c = c;
    w.neg = c < 0.0;
    const uint64_t cb = f64_bits(c) & 0x7FFFFFFFFFFFFFFFull;
    w.ac = bits_f64(cb);
    w.ec = (int) (cb >> 52);
    w.fast = w.ec >= 1023 - 23 && w.ec < 1023 + 9;      // 2^-23 <= |c| < 512
    w.rinv = w.fast ? (1.0 / w.ac) * (1.0 - 0x1p-29) : 0.0;
    return w;
}

// One iteration: jump as far as provably stays inside the current binade, then (if steps
// remain) one real step. `special` iterations (x below |c|, non-positive x, or an odd
// mantissa in a tie binade) jump zero steps. Returns true when the real step wrapped.
// floor of a non-negative double below 2^52, staying in the FP64 domain on the device
// (the step counter `nd` of the walk is kept as a double there: no int<->fp conversions on
// the loop-carried dependency chain)
GPSB_HD double floor_nonneg(double v) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(__dadd_rd(v, 0x1p52), -0x1p52);
#else
    return (double) (int64_t) v;
#endif
}

template <int KIND>
GPSB_HD bool walk_iteration(double &x, const WalkConst &w, double &nd, int64_t &periods, double *after_jump) {
    const uint64_t bx = f64_bits(x);
    const int ex = (int) ((bx >> 52) & 0x7FF);
    bool special = (bx >> 63) || !(x >= w.ac);
    const double lo = bits_f64((uint64_t) ex << 52);
    double stepd = (lo + w.ac) - lo;                    // |c| rounded to the grid of [2^e, 2^(e+1))
    if (ex == w.ec) stepd = w.ac;                       // own binade of c: steps are exact
    const double half_u = bits_f64((uint64_t) (ex > 53 ? ex - 53 : 0) << 52);
    const double res = w.ac - stepd;
    special |= ((res == half_u) | (res == -half_u)) & ((bx & 1) != 0);
    double room;
    if (!w.neg) {
        const uint64_t top = (KIND == NCO_CODE && ex == 1023 + 9) ? f64_bits(1023.0) : ((uint64_t) (ex + 1) << 52);
        room = bits_f64(top - 1) - x;                   // distance to the last double inside
    } else {
        room = x - lo;
    }
    double kq = room * w.rinv;
    if (kq > nd) kq = nd;
    if (special) kq = 0.0;
    const double k = floor_nonneg(kq);                  // integer-valued, <= nd < 2^31
    const double adv = k * stepd;                       // exact: k*R < 2^53
    x = w.neg ? x - adv : x + adv;                      // exact
    nd -= k;
    if (after_jump) *after_jump = x;
    bool wrapped = false;
    if (nd > 0.0) {
        const double before = x;
        nco_step<KIND>(x, w.c, periods);
        nd -= 1.0;
        wrapped = w.neg ? (x > before) : (x < before);
    }
    return wrapped;
}

// Advance x by exactly n reference steps of increment c (n < 2^31).
// Returns the number of loop iterations spent (diagnostics only).
template <int KIND>
GPSB_HD int nco_advance(double &x, double c, int64_t n, int64_t &periods) {
    if (c == 0.0 || n <= 0) return 0;
    const WalkConst w = walk_const(c);
    if (!w.fast || (KIND == NCO_CODE && w.neg)) return nco_advance_generic<KIND>(x, c, n, periods);
    int iters = 0;
    double nd = (double) n;
    while (nd > 0.0) {
        ++iters;
        walk_iteration<KIND>(x, w, nd, periods, nullptr);
    }
    return iters;
}

// ---------------------------------------------------------------------------------
// Parallel-in-time carrier chain: speculate per block, fix up sequentially.
//
// The carrier phase at the start of block b+1 is the end state of block b, a chain
// that is serial over the whole run. It is broken up with one property of the
// recurrence: if two trajectories of the SAME block (same c) have both just wrapped at
// the same sample, they differ by a multiple G of the coarsest rounding grid in play
// (G = 2^-52 for c > 0: results in [1,2) before the wrap subtraction; G = 2^-53 for
// c < 0), and from then on every rounding step commutes with that shift -- so the two
// stay exactly parallel -- as long as (1) they are in the same binade at every step,
// and (2) the shift is an EVEN multiple of G (an exact round-half-even tie resolves
// identically only then).
// carrier_probe() walks a block from a GUESSED start phase and reports: the sample
// index and state right after its first wrap; then, for both parities v (start state
// x_w and x_w + G), the end-of-block state and how far the trajectory could be shifted
// up/down without any visited state leaving its binade. carrier_fixup() (host, serial
// over blocks, a few jump iterations each) walks the TRUE start phase to that first
// wrap, picks the parity with an even shift, checks the shift against the margins and
// returns the exact end state -- or reports failure, in which case the caller falls
// back to the exact sequential walk nco_advance(). Either way the result is exact.
struct CarrierProbe {
    double x_w;          // guessed trajectory right after its first wrap
    double x_end[2];     // end-of-block state for start x_w + v*G
    double m_pos[2];     // largest upward shift tolerated (exclusive)
    double m_neg[2];     // largest downward shift tolerated (inclusive)
    int32_t n_w;         // steps done when the first wrap happened (1-based), -1: no wrap in the block
    int32_t pad;
};

GPSB_HD double carrier_grid(double c) { return c > 0.0 ? 0x1p-52 : 0x1p-53; }

// distance of v to the edges of its own binade [2^e, 2^(e+1)); 0 for v <= 0
GPSB_HD void binade_margins(double v, double &m_pos, double &m_neg) {
    const uint64_t b = f64_bits(v);
    if ((b >> 63) || (b >> 52) == 0) {
        m_pos = 0.0;
        m_neg = 0.0;
        return;
    }
    const double lo = bits_f64(b & 0xFFF0000000000000ull);
    const double up = (lo + lo) - v, dn = v - lo;
    if (up < m_pos) m_pos = up;
    if (dn < m_neg) m_neg = dn;
}

// Walk up to n steps like nco_advance<NCO_CARRIER>; stop right after the first wrap when
// stop_at_wrap; when margins are requested, fold every explicitly visited state (before the
// jump, after the jump, after the real step) into them. Returns the number of steps done.
// Degenerate increments (|c| < 2^-23) are not walked here: ok is cleared and the caller
// treats the block as "no usable speculation".
GPSB_HD int64_t carrier_walk_w(double &x, const WalkConst &w, int64_t n, bool stop_at_wrap, bool &wrapped, bool &ok,
                               double *m_pos, double *m_neg) {
    wrapped = false;
    ok = true;
    if (n <= 0) return 0;
    if (w.c == 0.0 || !w.fast) {
        ok = false;
        return 0;
    }
    const double n0 = (double) n;
    double nd = n0;
    int64_t dummy = 0;
    if (m_pos) binade_margins(x, *m_pos, *m_neg);       // start state; later loop-top states were folded in
    while (nd > 0.0) {                                   // as the previous iteration's post-step state
        double aj;
        const bool wr = walk_iteration<NCO_CARRIER>(x, w, nd, dummy, &aj);
        if (m_pos) {
            binade_margins(aj, *m_pos, *m_neg);
            binade_margins(x, *m_pos, *m_neg);
        }
        if (wr) {
            wrapped = true;
            if (stop_at_wrap) break;
        }
    }
    return (int64_t) (n0 - nd);
}

GPSB_HD int64_t carrier_walk(double &x, double c, int64_t n, bool stop_at_wrap, bool &wrapped, bool &ok,
                             double *m_pos, double *m_neg) {
    const WalkConst w = walk_const(c);
    return carrier_walk_w(x, w, n, stop_at_wrap, wrapped, ok, m_pos, m_neg);
}

// One parity variant v of the probe (the device runs the two variants in different threads;
// each repeats the short walk to the first wrap). Fills n_w/x_w (identical for both v) and
// the v-th end state and margins.
GPSB_HD void carrier_probe_variant(double guess, double c, int64_t n, int v, CarrierProbe &o) {
    double x = guess;
    bool wrapped = false, ok = true;
    const int64_t nw = carrier_walk(x, c, n, true, wrapped, ok, nullptr, nullptr);
    o.pad = 0;
    if (!wrapped || !ok) {
        o.n_w = -1;
        o.x_w = x;
        o.x_end[v] = x;
        o.m_pos[v] = o.m_neg[v] = 0.0;
        return;
    }
    o.n_w = (int32_t) nw;
    o.x_w = x;
    double xv = x + (v ? carrier_grid(c) : 0.0);       // exact: x_w is a multiple of G
    double mp = 1.0, mn = 1.0;
    bool w2, ok2;
    // a parity partner that left [0,1) (x_w at the very edge) is simply unusable
    if (!(xv >= 0.0 && xv < 1.0)) mp = mn = 0.0;
    else carrier_walk(xv, c, n - nw, false, w2, ok2, &mp, &mn);
    o.x_end[v] = xv;
    o.m_pos[v] = mp;
    o.m_neg[v] = mn;
}

GPSB_HD void carrier_probe(double guess, double c, int64_t n, CarrierProbe &o) {
    carrier_probe_variant(guess, c, n, 0, o);
    carrier_probe_variant(guess, c, n, 1, o);
}

// Exact end-of-block carrier phase from the true start s and the probe of a guessed start.
// Returns false when the speculation cannot be used (caller then runs nco_advance).
// v_out / d_out (optional): the parity variant chosen and the shift of the true trajectory against it;
// `safety` scales the margins (0.5 for a block probe: half the measured room; 1.0 for a span summary whose
// margins are already net of the safety factor and of the per-block shifts, see span_chain()).
// pre_mp / pre_mn (optional): binade margins of the states the walk from s to the first wrap visited -- how far
// THAT piece of trajectory could itself be shifted (span_chain() walks a speculative start here).
GPSB_HD bool carrier_fixup(double s, double c, const CarrierProbe &p, double &x_end, int *v_out = nullptr,
                           double *d_out = nullptr, double safety = 0.5, double *pre_mp = nullptr,
                           double *pre_mn = nullptr) {
    if (p.n_w < 0) return false;
    double a = s;
    bool wrapped = false, ok = true;
    if (pre_mp) *pre_mp = *pre_mn = 1.0;
    // the true trajectory must wrap for the first time exactly at step n_w
    const int64_t done = carrier_walk(a, c, p.n_w, true, wrapped, ok, pre_mp, pre_mn);
    if (!ok || !wrapped || done != p.n_w) return false;
    const double G = carrier_grid(c);
    const double d0 = a - p.x_w;                        // exact: both multiples of G, both small
    const double q = d0 / G;                            // exact scaling by a power of two
    if (!(q > -0x1p40 && q < 0x1p40)) return false;
    const long long qi = (long long) q;
    if ((double) qi != q) return false;
    const int v = (int) (qi & 1);
    const double d = d0 - (v ? G : 0.0);                // even multiple of G
    // half the measured room as a safety factor (margins are ~1e-7, shifts ~1e-12)
    if (!(d < safety * p.m_pos[v] && -d < safety * p.m_neg[v])) return false;
    x_end = p.x_end[v] + d;                             // exact: the sum IS the true state
    if (v_out) *v_out = v;
    if (d_out) *d_out = d;
    return true;
}

// ---------------------------------------------------------------------------------------------------
// Second level of the parallel-in-time chain: SPANS of consecutive blocks.
//
// Once two trajectories of one satellite differ by an even multiple of G they stay exactly parallel ACROSS
// block boundaries too (the increment changes, the argument of carrier_probe() does not: the shift is a
// multiple of every rounding grid in play, ties resolve identically) -- as long as they share the binade
// at every step and the sign of the increment (hence G) does not change. So a whole span of K blocks can be
// resolved SPECULATIVELY on the device: span_chain() chains the K block probes from the span's guessed
// start phase exactly like the host scan does, once per parity variant V of the first block, and records
// the speculative start phase of every block plus how far the whole speculative trajectory may still be
// shifted. The result is a CarrierProbe for the span as a whole: the host turns the TRUE start phase of
// the span into the true end phase with ONE carrier_fixup() (safety 1.0) -- K times fewer serial links --
// and the true start phase of block j is the speculative one plus the span's shift D.
// A span is REGULAR when one satellite holds the slot in all its blocks, every increment has the same
// sign (and is not 0), the first block wraps, and every block probe could be used; otherwise (reallocation
// inside the span, Doppler zero crossing, a rejected probe: all rare) ok = 0 and the host resolves that
// span block by block from the block probes.
struct SpanBlockState {      // per (block, channel), for the span's variants V = 0, 1:
    double start[2];         // speculative start phase of the block
};

// probes / blocks: element j of the span lives at index j * stride; param(j, c, prn) yields block j's carrier
// increment and satellite.
template <class ParamFn>
GPSB_HD void span_chain(const CarrierProbe *probes, ParamFn param, int nblk_span, size_t stride, double guess, int V,
                        CarrierProbe &sum, bool &ok, SpanBlockState *blocks) {
    ok = false;
    sum.n_w = -1;
    sum.pad = 0;
    sum.x_w = 0.0;
    sum.x_end[V] = sum.m_pos[V] = sum.m_neg[V] = 0.0;
    const CarrierProbe &p0 = probes[0];
    blocks[0].start[V] = guess;
    double c0;
    int32_t prn0;
    param(0, c0, prn0);
    if (prn0 <= 0 || p0.n_w < 0 || c0 == 0.0) return;
    const bool neg = c0 < 0.0;
    double x = p0.x_end[V];
    double mp = 0.5 * p0.m_pos[V], mn = 0.5 * p0.m_neg[V];
    if (!(mp > 0.0 && mn > 0.0)) return;
    for (int j = 1; j < nblk_span; j++) {
        const size_t i = (size_t) j * stride;
        blocks[i].start[V] = x;
        double c;
        int32_t prn;
        param(j, c, prn);
        if (prn != prn0 || c == 0.0 || (c < 0.0) != neg) return;
        int v;
        double d, xe, pmp, pmn;
        if (!carrier_fixup(x, c, probes[i], xe, &v, &d, 0.5, &pmp, &pmn)) return;
        // room left for a further shift D of the whole speculative trajectory: after the block's first wrap the
        // block probe's margins net of this block's own shift d, before it the margins of the walk just done
        const double a = 0.5 * probes[i].m_pos[v] - d, b = 0.5 * probes[i].m_neg[v] + d;
        if (a < mp) mp = a;
        if (b < mn) mn = b;
        if (0.5 * pmp < mp) mp = 0.5 * pmp;
        if (0.5 * pmn < mn) mn = 0.5 * pmn;
        x = xe;
    }
    sum.n_w = p0.n_w;
    sum.x_w = p0.x_w;
    sum.x_end[V] = x;
    sum.m_pos[V] = mp;
    sum.m_neg[V] = mn;
    ok = true;
}

// Expected rounding drift per step of the carrier recurrence (host only): while the phase
// sweeps [0,1) uniformly it spends a fraction 2^e of the steps in binade [2^e, 2^(e+1)),
// where each step really adds R_e*u_e instead of c. Used to GUESS block-start phases for
// carrier_probe(); accuracy only affects how often carrier_fixup() must fall back.
inline double carrier_drift_per_step(double c) {
    if (c == 0.0) return 0.0;
    const uint64_t cb = f64_bits(c) & 0x7FFFFFFFFFFFFFFFull;
    const int ec = (int) (cb >> 52);
    if (ec == 0 || ec >= 1022) return 0.0;
    const double ac = bits_f64(cb);
    // In binade [2^e, 2^(e+1)) a step adds |c| rounded to that binade's grid, which FP64 itself yields as
    // (2^e + |c|) - 2^e (round-half-even == the even neighbour once the mantissa is even); the binade is
    // visited a fraction 2^e of the time.
    double tot = 0.0;
    for (int ex = ec + 1; ex <= 1022; ex++) {           // up to the binade [0.5, 1)
        if (ex - ec >= 54) break;
        const double lo = bits_f64((uint64_t) ex << 52);
        const double stepd = (lo + ac) - lo;
        tot += (stepd - ac) * lo;                       // exact difference, weight 2^e
    }
    return c > 0.0 ? tot : -tot;
}

// NAV-message position after `periods` more code periods (gps.c:2793-2812):
// 20 code periods per data bit, 30 bits per word.
GPSB_HD void nav_advance(int &iword, int &ibit, int &icode, int64_t periods) {
    int64_t t = (int64_t) icode + periods;
    icode = (int) (t % 20);
    t = (int64_t) ibit + t / 20;
    ibit = (int) (t % 30);
    iword += (int) (t / 30);
}

}  // namespace gpsb200
