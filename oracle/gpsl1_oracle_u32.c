/* TEST INFRASTRUCTURE -- parity oracle of the reference's INTEGER carrier build, not product code.
 *
 * The reference's sample loop has two builds, selected by `#define FLOAT_CARR_PHASE` (gps.h:17). Without it the
 * carrier NCO is an unsigned 32-bit accumulator: carr_phasestep = (int) round(512.0 * 65536.0 * f_carr * delt) once
 * per block (gps.c:2745-2747), table index (carr_phase >> 16) & 511 (gps.c:2777), carr_phase += carr_phasestep modulo
 * 2^32 after every sample (gps.c:2828). Everything else (code NCO, NAV bits, tables, accumulation) is the FP64 build's,
 * see gpsl1_oracle.c. Linked into liboracle_gpsl1_u32.so together with gpsl1_oracle.c (oracle/u32.mk). */
#include <math.h>
#include <stdlib.h>
#include "gpsl1_oracle.h"

/* Same record as oracle_synth_block; carr_phase holds the u32 accumulator as an integer-valued double in
 * [0, 2^32) and is left as the loop leaves it. */
void oracle_synth_block_u32(oracle_chan_t *ch, int nchan, int nsamp, int16_t *iq16) {
    const double delt = 1.0 / 3000000.0;       /* gps.c:2298, sdr.h:21 */
    int32_t *acc = calloc((size_t) 2 * nsamp, sizeof *acc);
    int32_t s512[512], c512[512];
    oracle_tables(s512, c512);

    for (int c = 0; c < nchan; c++) {
        oracle_chan_t *p = &ch[c];
        if (p->prn <= 0) continue;
        uint8_t ca[ORACLE_CA_LEN];
        oracle_codegen(p->prn, ca);
        int32_t ai[512], aq[512];
        for (int k = 0; k < 512; k++) {        /* gps.c:2781-2782 */
            ai[k] = (int32_t) ((double) c512[k] * p->gain);
            aq[k] = (int32_t) ((double) s512[k] * p->gain);
        }
        /* gps.c:2746: left to right, (512.0 * 65536.0) folded by the compiler, C round (ties away from zero) */
        const int step = (int) round(512.0 * 65536.0 * p->f_carr * delt);
        const double dcode = p->f_code * delt; /* gps.c:2789 */
        unsigned int carr = (unsigned int) p->carr_phase;
        double code = p->code_phase;
        int iword = p->iword, ibit = p->ibit, icode = p->icode;
        int bit = (int) ((p->dwrd[iword] >> (29 - ibit)) & 1u);
        for (int n = 0; n < nsamp; n++) {
            const int k = (carr >> 16) & 511;                     /* gps.c:2777 */
            const int sign = (bit == ca[(int) code]) ? 1 : -1;
            acc[2 * n] += sign * ai[k];
            acc[2 * n + 1] += sign * aq[k];

            code += dcode;                                        /* gps.c:2789-2817 */
            if (code >= 1023.0) {
                code -= 1023.0;
                if (++icode >= 20) {
                    icode = 0;
                    if (++ibit >= 30) { ibit = 0; iword++; }
                    bit = (int) ((p->dwrd[iword] >> (29 - ibit)) & 1u);
                }
            }
            carr += (unsigned int) step;                          /* gps.c:2828, modulo 2^32 */
        }
        p->carr_phase = (double) carr; p->code_phase = code;
        p->iword = iword; p->ibit = ibit; p->icode = icode;
    }
    for (int j = 0; j < 2 * nsamp; j++) iq16[j] = (int16_t) acc[j];
    free(acc);
}
