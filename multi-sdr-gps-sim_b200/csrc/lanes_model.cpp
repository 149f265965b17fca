// Host model of the LANE = SAMPLE synthesis (synth_lanes.h): the same window / band / repair logic the CUDA kernel
// k_synth_lanes runs, executed sample by sample on the CPU for ONE block. Exists so that the algorithm's exactness can
// be tested against the oracle without a GPU (tests/test_host_api.py); it is not a product path and nothing calls it
// except the tests.
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/gpsb200.h"
#include "nco_exact.h"
#include "synth_lanes.h"
#include "synth_tables.h"

using namespace gpsb200;

namespace {
int sine512_host(int k) {
    static const uint8_t q[128] = {GPSB200_QUARTER_SINE};
    k &= 511;
    const int r = k & 255;
    const int v = q[r < 128 ? r : 255 - r];
    return k < 256 ? v : -v;
}
}  // namespace

extern "C" int gpsb200_lanes_model_block(const gpsb200_chan_t *chans, int nchan, const uint32_t *nav /* [nchan][60] */,
                                         int run_samples, int force, int16_t *iq /* [600000] */, double *carr_out,
                                         int64_t *counters /* [4]: fast, repaired samples, slow windows, walks */) {
    if (!chans || !nav || !iq || nchan < 1 || nchan > 32 || run_samples % lanes::kWindow != 0 || run_samples > lanes::kMaxRun ||
        GPSB200_BLOCK_SAMPLES % run_samples != 0)
        return GPSB200_ERR_ARG;
    const double delt = 1.0 / (double) GPSB200_SAMPLERATE;
    const bool u32 = (force & 16) != 0;          // GPSB200_CARRIER_U32: exact phases, as k_synth_lanes<.., U32 = true>
    const int nruns = GPSB200_BLOCK_SAMPLES / run_samples, nwin = run_samples / lanes::kWindow;
    std::vector<std::vector<uint32_t>> chipw(nchan, std::vector<uint32_t>(36, 0));
    std::vector<std::vector<int32_t>> tab(nchan, std::vector<int32_t>(512, 0));
    for (int c = 0; c < nchan; c++) {
        if (chans[c].prn <= 0) continue;
        if (u32 && !(chans[c].carr_phase >= 0.0 && chans[c].carr_phase < 4294967296.0 &&
                     chans[c].carr_phase == std::floor(chans[c].carr_phase)))
            return GPSB200_ERR_ARG;
        if (!lanes::code_step_ok(chans[c].f_code * delt)) return GPSB200_ERR_RANGE;
        uint8_t ca[GPSB200_CA_LEN];
        ca_code(chans[c].prn, ca);
        for (int n = 0; n < 36 * 32; n++)
            if (ca[n % GPSB200_CA_LEN]) chipw[c][n >> 5] |= 1u << (n & 31);
        for (int k = 0; k < 512; k++) {                                      // gps.c:2781-2782
            const int ai = (int) ((double) sine512_host(k + 128) * chans[c].gain);
            const int aq = (int) ((double) sine512_host(k) * chans[c].gain);
            tab[c][k] = ai + aq * 65536;
        }
    }
    int64_t cnt[4] = {0, 0, 0, 0};
    std::vector<double> x(nchan), y(nchan);
    std::vector<int> iword(nchan), ibit(nchan), icode(nchan);
    for (int c = 0; c < nchan; c++) {
        x[c] = chans[c].carr_phase;
        y[c] = chans[c].code_phase;
        iword[c] = chans[c].iword;
        ibit[c] = chans[c].ibit;
        icode[c] = chans[c].icode;
    }
    std::vector<lanes::ChanRun> st(nchan);
    std::vector<lanes::Anchor> an(nchan);
    for (int r = 0; r < nruns; r++) {
        for (int c = 0; c < nchan; c++) {
            const uint32_t *nv = nav + (size_t) c * 60;
            auto navf = [nv](int iw) { return nv[iw]; };
            const uint32_t pos = (uint32_t) iword[c] | ((uint32_t) ibit[c] << 8) | ((uint32_t) icode[c] << 16);
            an[c] = lanes::Anchor{x[c], y[c], chans[c].f_carr * delt, chans[c].f_code * delt, pos};
            lanes::init_run(st[c], chans[c].prn > 0, x[c], y[c], pos, an[c].c, an[c].d, navf);
        }
        for (int w = 0; w < nwin; w++) {
            std::vector<uint32_t> S(3 * nchan, 0), base(nchan, 0), step(nchan, 0);
            for (int c = 0; c < nchan; c++) {
                if (!st[c].active) continue;
                const uint32_t *nv = nav + (size_t) c * 60;
                auto navf = [nv](int iw) { return nv[iw]; };
                const uint32_t *cw = chipw[c].data();
                auto chipf = [cw](int i) { return cw[i]; };
                const bool ok = lanes::window_signs(st[c], chipf, navf, &S[3 * c], (force & 8) != 0);
                if (!ok || (force & 2)) {
                    lanes::exact_signs(an[c], w, chipf, navf, &S[3 * c]);
                    ++cnt[2];
                }
                if (u32) {       // window record of the U32 variant: (u_run + 96 w step) << 7, step << 7
                    const uint32_t su = (uint32_t) lanes::u32_carrier_step(chans[c].f_carr);
                    base[c] = ((uint32_t) x[c] + (uint32_t) (w * lanes::kWindow) * su) << 7;
                    step[c] = su << 7;
                } else {
                    base[c] = lanes::fast_base(st[c]);
                    step[c] = lanes::fast_step(st[c]);
                }
            }
            for (int n = 0; n < lanes::kWindow; n++) {
                const int q = n / 3, rr = n - 3 * q;
                int acc = 0;
                bool repaired = false;
                for (int c = 0; c < nchan; c++) {
                    if (!st[c].active) continue;
                    const uint32_t p = base[c] + (uint32_t) n * step[c];
                    int k = (int) (p >> 23);
                    if (!u32 && (lanes::fast_risky(p) || (force & 1))) {
                        const uint64_t m = st[c].P + (uint64_t) n * st[c].D;
                        const uint64_t frac = m & ((1ull << 55) - 1);
                        if ((force & 4) || frac < lanes::kBandCarr || frac > (1ull << 55) - lanes::kBandCarr) ++cnt[3];
                        k = lanes::exact_index(st[c].P, st[c].D, an[c], w, n, (force & 4) != 0);
                        repaired = true;
                    }
                    const int sign = (int) ((S[3 * c + rr] >> q) & 1u);
                    acc += tab[c][k ^ (sign << 8)];                       // table[k ^ 256] = -table[k]
                }
                ++cnt[repaired ? 1 : 0];
                const int iv = (int) (short) (acc & 0xFFFF), qv = (acc - iv) >> 16;
                const size_t o = ((size_t) r * run_samples + (size_t) w * lanes::kWindow + n) * 2;
                iq[o] = (int16_t) iv;
                iq[o + 1] = (int16_t) qv;
            }
            for (int c = 0; c < nchan; c++) {
                if (!st[c].active) continue;
                const uint32_t *nv = nav + (size_t) c * 60;
                lanes::advance_window(st[c], [nv](int iw) { return nv[iw]; });
            }
        }
        // exact anchors of the next run (what k_checkpoints provides on the device)
        for (int c = 0; c < nchan; c++) {
            if (chans[c].prn <= 0) continue;
            int64_t periods = 0, dummy = 0;
            if (u32) x[c] = (double) ((uint32_t) x[c] + (uint32_t) run_samples * (uint32_t) lanes::u32_carrier_step(chans[c].f_carr));
            else nco_advance<NCO_CARRIER>(x[c], chans[c].f_carr * delt, run_samples, dummy);
            nco_advance<NCO_CODE>(y[c], chans[c].f_code * delt, run_samples, periods);
            nav_advance(iword[c], ibit[c], icode[c], periods);
        }
    }
    if (carr_out)
        for (int c = 0; c < nchan; c++) carr_out[c] = chans[c].prn > 0 ? x[c] : 0.0;
    if (counters) memcpy(counters, cnt, sizeof cnt);
    return GPSB200_OK;
}
