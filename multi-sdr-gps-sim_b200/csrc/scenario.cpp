// Host-side scenario engine: RINEX-2 navigation file + receiver location/motion ->
// per-block channel parameters (gpsb200_chan_t) and NAV frames, i.e. everything the
// reference's producer thread computes OUTSIDE its sample loop:
//   RINEX v2 / v3 readers      (reference gps.c:1131-1505, 1512-1891)
//   time / coordinate helpers  (gps.c:315-499, 1094-1124)
//   satellite position, range, Klobuchar delay (gps.c:508-611, 1893-2026)
//   code phase / NAV position  (gps.c:2033-2064)
//   subframes, parity, 30 s NAV frames (gps.c:617-884, 1008-1072, 2066-2140)
//   visibility + channel allocation (gps.c:2142-2235), 10 Hz loop (gps.c:2703-2765, 2870-2932)
// These are rows f1/f2/f4 of SURVEY.md section 8 ("next" after the sample loop). The
// doubles feed the CUDA kernels bit for bit, so every expression keeps the reference's
// evaluation order (no FMA contraction: -ffp-contract=off) and the same libm calls;
// tests/test_scenario.py compares every field with the reference's own dumps.
//
//   SEM almanac reader + almanac pages of subframes 4/5 (almanac.c:73-184, gps.c:772-884),
//   when a local almanac file is given (the reference's almanac.sem; none = its almanac disabled)
//
// Scope notes: almanac downloads (-f), RINEX downloads, interactive motion and
// the HackRF/Pluto specifics (except the Pluto gain doubling) are out of scope.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include <zlib.h>

#include "../../include/gpsb200.h"
#include "synth_tables.h"

namespace {

// ---- constants of the reference (gps.h:60-118) --------------------------------------
constexpr double kSecWeek = 604800.0, kSecHalfWeek = 302400.0, kSecDay = 86400.0, kSecHour = 3600.0;
constexpr double kGM = 3.986005e14, kOmegaE = 7.2921151467e-5, kPi = 3.1415926535898;
constexpr double kWgsA = 6378137.0, kWgsE = 0.0818191908426, kR2D = 57.2957795131;
constexpr double kC = 2.99792458e8, kLambda = 0.190293672798365;
constexpr double kCodeFreq = 1.023e6, kCarrToCode = 1.0 / 1540.0;
constexpr int kMaxSat = 32, kEphSets = 13, kSbfPages = 3 + 2 * 25, kWordsPerSbf = 10;
// 2^-n scale factors exactly as spelled in gps.h:66-83 (the literals, not ldexp: a few of
// them differ from the true power of two in the last digits)
constexpr double P2_5 = 0.03125, P2_19 = 1.907348632812500e-6, P2_29 = 1.862645149230957e-9,
                 P2_31 = 4.656612873077393e-10, P2_33 = 1.164153218269348e-10, P2_43 = 1.136868377216160e-13,
                 P2_55 = 2.775557561562891e-17, P2_50 = 8.881784197001252e-016, P2_30 = 9.313225746154785e-010,
                 P2_27 = 7.450580596923828e-009, P2_24 = 5.960464477539063e-008;
// the almanac's scale factors (gps.h:79-84); P2_38 and P2_23 are not exact powers of two, and 2^12 is an int there
constexpr double P2_21 = 4.76837158203125e-007, P2_38 = 3.63797880709171e-012, P2_11 = 0.00048828125,
                 P2_23 = 1.19209289550781e-007, P2_20 = 9.5367431640625e-007;
constexpr int P2p12 = 4096;
// receiver antenna attenuation in dB per 5 deg of boresight angle (gps.c:215-220)
const double kAntPatDb[37] = {0.00,  0.00,  0.22,  0.44,  0.67,  1.11,  1.56,  2.00,  2.44,  2.89,  3.56,  4.22,  4.89,
                              5.56,  6.22,  6.89,  7.56,  8.22,  8.89,  9.78,  10.67, 11.56, 12.44, 13.33, 14.44, 15.56,
                              16.67, 17.78, 18.89, 20.00, 21.33, 22.67, 24.00, 25.56, 27.33, 29.33, 31.56};

struct GpsTime {
    int week = 0;
    double sec = 0.0;
};
struct Date {
    int y = 0, m = 0, d = 0, hh = 0, mm = 0;
    double sec = 0.0;
};
struct Eph {
    bool valid = false;
    int svh = 0, iodc = 0, iode = 0;
    Date t;
    GpsTime toc, toe;
    double deltan = 0, cuc = 0, cus = 0, cic = 0, cis = 0, crc = 0, crs = 0, ecc = 0, sqrta = 0, m0 = 0, omg0 = 0,
           inc0 = 0, aop = 0, omgdot = 0, idot = 0, af0 = 0, af1 = 0, af2 = 0, tgd = 0;
    double n = 0, sq1e2 = 0, A = 0, omgkdot = 0;      // derived (gps.c:1489-1493)
};
struct IonoUtc {
    bool enable = true, valid = false;
    double alpha[4] = {0, 0, 0, 0}, beta[4] = {0, 0, 0, 0}, A0 = 0, A1 = 0;
    int dtls = 0, tot = 0, wnt = 0;
};
struct Range {
    GpsTime g;
    double range = 0, rate = 0, d = 0, az = 0, el = 0, iono = 0;
};
struct Channel {
    int prn = 0;
    double f_carr = 0, f_code = 0, carr_phase = 0, code_phase = 0;
    GpsTime g0;
    uint32_t sbf[kSbfPages][kWordsPerSbf];
    uint32_t dwrd[GPSB200_NAV_WORDS];
    int ipage = 0, iword = 0, ibit = 0, icode = 0;
    Range rho0;
};
// one SEM almanac record (almanac.h:21-37): angles in semicircles, as the file gives them
struct AlmanacSv {
    unsigned char ura = 0, health = 0, config_code = 0;
    unsigned short svid = 0, svn = 0;       // svid != 0: the record was started (its ID line was read)
    unsigned valid = 0;                     // 1: the record was read to its end
    double e = 0, delta_i = 0, omegadot = 0, sqrta = 0, omega0 = 0, aop = 0, m0 = 0, af0 = 0, af1 = 0;
    GpsTime toa;                            // set only when the record is complete
};
struct Almanac {
    unsigned valid = 0;                     // at least one complete record
    AlmanacSv sv[kMaxSat];
};

// ---- time (gps.c:315-339, 1094-1124) ---------------------------------------------------
GpsTime date_to_gps(const Date &t) {
    static const int doy[12] = {0, 31, 59, 90, 120, 151, 181, 212, 243, 273, 304, 334};
    const int ye = t.y - 1980;
    int lpdays = ye / 4 + 1;
    if ((ye % 4) == 0 && t.m <= 2) lpdays--;
    const int de = ye * 365 + doy[t.m - 1] + t.d + lpdays - 6;
    GpsTime g;
    g.week = de / 7;
    g.sec = (double) (de % 7) * kSecDay + t.hh * kSecHour + t.mm * 60.0 + t.sec;
    return g;
}
double gps_diff(const GpsTime &a, const GpsTime &b) {
    double dt = a.sec - b.sec;
    dt += (double) (a.week - b.week) * kSecWeek;
    return dt;
}
GpsTime gps_add(const GpsTime &g0, double dt) {
    GpsTime g = g0;
    g.sec = g0.sec + dt;
    g.sec = round(g.sec * 1000.0) / 1000.0;
    while (g.sec >= kSecWeek) {
        g.sec -= kSecWeek;
        g.week++;
    }
    while (g.sec < 0.0) {
        g.sec += kSecWeek;
        g.week--;
    }
    return g;
}

// ---- coordinates (gps.c:361-499) ----------------------------------------------------------
double norm3(const double *v) { return sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); }
double dot3(const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

void ecef_to_llh(const double *xyz, double *llh) {
    const double a = kWgsA, e = kWgsE, eps = 1.0e-3, e2 = e * e;
    if (norm3(xyz) < eps) {
        llh[0] = 0.0;
        llh[1] = 0.0;
        llh[2] = -a;
        return;
    }
    const double x = xyz[0], y = xyz[1], z = xyz[2];
    const double rho2 = x * x + y * y;
    double dz = e2 * z, zdz, nh, slat, n;
    for (;;) {
        zdz = z + dz;
        nh = sqrt(rho2 + zdz * zdz);
        slat = zdz / nh;
        n = a / sqrt(1.0 - e2 * slat * slat);
        const double dz_new = n * e2 * slat;
        if (fabs(dz - dz_new) < eps) break;
        dz = dz_new;
    }
    llh[0] = atan2(zdz, sqrt(rho2));
    llh[1] = atan2(y, x);
    llh[2] = nh - n;
}
void llh_to_ecef(const double *llh, double *xyz) {
    const double a = kWgsA, e = kWgsE, e2 = e * e;
    const double clat = cos(llh[0]), slat = sin(llh[0]), clon = cos(llh[1]), slon = sin(llh[1]);
    const double d = e * slat;
    const double n = a / sqrt(1.0 - d * d);
    const double nph = n + llh[2];
    const double tmp = nph * clat;
    xyz[0] = tmp * clon;
    xyz[1] = tmp * slon;
    xyz[2] = ((1.0 - e2) * n + llh[2]) * slat;
}
void local_frame(const double *llh, double t[3][3]) {
    const double slat = sin(llh[0]), clat = cos(llh[0]), slon = sin(llh[1]), clon = cos(llh[1]);
    t[0][0] = -slat * clon;
    t[0][1] = -slat * slon;
    t[0][2] = clat;
    t[1][0] = -slon;
    t[1][1] = clon;
    t[1][2] = 0.0;
    t[2][0] = clat * clon;
    t[2][1] = clat * slon;
    t[2][2] = slat;
}
void az_el(const double *los, const double t[3][3], double &az, double &el) {
    double neu[3];
    for (int i = 0; i < 3; i++) neu[i] = t[i][0] * los[0] + t[i][1] * los[1] + t[i][2] * los[2];
    az = atan2(neu[1], neu[0]);
    if (az < 0.0) az += (2.0 * kPi);
    const double ne = sqrt(neu[0] * neu[0] + neu[1] * neu[1]);
    el = atan2(neu[2], ne);
}

// ---- satellite position / velocity / clock (gps.c:508-611) -----------------------------------
void sat_state(const Eph &e, const GpsTime &g, double *pos, double *vel, double *clk) {
    double tk = g.sec - e.toe.sec;
    if (tk > kSecHalfWeek) tk -= kSecWeek;
    else if (tk < -kSecHalfWeek) tk += kSecWeek;
    const double mk = e.m0 + e.n * tk;
    double ek = mk, ekold = ek + 1.0, one_m_ecosE = 0;
    while (fabs(ek - ekold) > 1.0E-14) {
        ekold = ek;
        one_m_ecosE = 1.0 - e.ecc * cos(ekold);
        ek = ek + (mk - ekold + e.ecc * sin(ekold)) / one_m_ecosE;
    }
    const double sek = sin(ek), cek = cos(ek);
    const double ekdot = e.n / one_m_ecosE;
    const double relativistic = -4.442807633E-10 * e.ecc * e.sqrta * sek;
    const double pk = atan2(e.sq1e2 * sek, cek - e.ecc) + e.aop;
    const double pkdot = e.sq1e2 * ekdot / one_m_ecosE;
    const double s2pk = sin(2.0 * pk), c2pk = cos(2.0 * pk);
    const double uk = pk + e.cus * s2pk + e.cuc * c2pk;
    const double suk = sin(uk), cuk = cos(uk);
    const double ukdot = pkdot * (1.0 + 2.0 * (e.cus * c2pk - e.cuc * s2pk));
    const double rk = e.A * one_m_ecosE + e.crc * c2pk + e.crs * s2pk;
    const double rkdot = e.A * e.ecc * sek * ekdot + 2.0 * pkdot * (e.crs * c2pk - e.crc * s2pk);
    const double ik = e.inc0 + e.idot * tk + e.cic * c2pk + e.cis * s2pk;
    const double sik = sin(ik), cik = cos(ik);
    const double ikdot = e.idot + 2.0 * pkdot * (e.cis * c2pk - e.cic * s2pk);
    const double xpk = rk * cuk, ypk = rk * suk;
    const double xpkdot = rkdot * cuk - ypk * ukdot, ypkdot = rkdot * suk + xpk * ukdot;
    const double ok = e.omg0 + tk * e.omgkdot - kOmegaE * e.toe.sec;
    const double sok = sin(ok), cok = cos(ok);
    pos[0] = xpk * cok - ypk * cik * sok;
    pos[1] = xpk * sok + ypk * cik * cok;
    pos[2] = ypk * sik;
    const double tmp = ypkdot * cik - ypk * sik * ikdot;
    vel[0] = -e.omgkdot * pos[1] + xpkdot * cok - tmp * sok;
    vel[1] = e.omgkdot * pos[0] + xpkdot * sok + tmp * cok;
    vel[2] = ypk * cik * ikdot + ypkdot * sik;
    tk = g.sec - e.toc.sec;
    if (tk > kSecHalfWeek) tk -= kSecWeek;
    else if (tk < -kSecHalfWeek) tk += kSecWeek;
    clk[0] = e.af0 + tk * (e.af1 + tk * e.af2) + relativistic - e.tgd;
    clk[1] = e.af1 + 2.0 * tk * e.af2;
}

// ---- Klobuchar ionospheric delay (gps.c:1893-1964) ----------------------------------------------
double iono_delay(const IonoUtc &io, const GpsTime &g, const double *llh, double az, double el) {
    if (!io.enable) return 0.0;
    const double E = el / kPi, phi_u = llh[0] / kPi, lam_u = llh[1] / kPi;
    const double F = 1.0 + 16.0 * pow((0.53 - E), 3.0);
    if (!io.valid) return F * 5.0e-9 * kC;
    const double psi = 0.0137 / (E + 0.11) - 0.022;
    double phi_i = phi_u + psi * cos(az);
    if (phi_i > 0.416) phi_i = 0.416;
    else if (phi_i < -0.416) phi_i = -0.416;
    const double lam_i = lam_u + psi * sin(az) / cos(phi_i * kPi);
    const double phi_m = phi_i + 0.064 * cos((lam_i - 1.617) * kPi);
    const double phi_m2 = phi_m * phi_m, phi_m3 = phi_m2 * phi_m;
    double AMP = io.alpha[0] + io.alpha[1] * phi_m + io.alpha[2] * phi_m2 + io.alpha[3] * phi_m3;
    if (AMP < 0.0) AMP = 0.0;
    double PER = io.beta[0] + io.beta[1] * phi_m + io.beta[2] * phi_m2 + io.beta[3] * phi_m3;
    if (PER < 72000.0) PER = 72000.0;
    double t = kSecDay / 2.0 * lam_i + g.sec;
    while (t >= kSecDay) t -= kSecDay;
    while (t < 0) t += kSecDay;
    const double X = 2.0 * kPi * (t - 50400.0) / PER;
    if (fabs(X) < 1.57) {
        const double X2 = X * X, X4 = X2 * X2;
        return F * (5.0e-9 + AMP * (1.0 - X2 / 2.0 + X4 / 24.0)) * kC;
    }
    return F * 5.0e-9 * kC;
}

// ---- pseudorange (gps.c:1972-2026) ------------------------------------------------------------------
Range pseudo_range(const Eph &e, const IonoUtc &io, const GpsTime &g, const double *xyz) {
    double pos[3], vel[3], clk[2], los[3];
    sat_state(e, g, pos, vel, clk);
    for (int i = 0; i < 3; i++) los[i] = pos[i] - xyz[i];
    const double tau = norm3(los) / kC;
    pos[0] -= vel[0] * tau;
    pos[1] -= vel[1] * tau;
    pos[2] -= vel[2] * tau;
    const double xrot = pos[0] + pos[1] * kOmegaE * tau;
    const double yrot = pos[1] - pos[0] * kOmegaE * tau;
    pos[0] = xrot;
    pos[1] = yrot;
    for (int i = 0; i < 3; i++) los[i] = pos[i] - xyz[i];
    Range r;
    const double range = norm3(los);
    r.d = range;
    r.range = range - kC * clk[0];
    r.rate = dot3(vel, los) / range;
    r.g = g;
    double llh[3], tm[3][3];
    ecef_to_llh(xyz, llh);
    local_frame(llh, tm);
    az_el(los, tm, r.az, r.el);
    r.iono = iono_delay(io, g, llh, r.az, r.el);
    r.range += r.iono;
    return r;
}

// ---- NAV words (gps.c:890-905, 1008-1072) -------------------------------------------------------------
unsigned parity_of(uint32_t v) { return (unsigned) __builtin_popcount(v) & 1u; }

// 30-bit word with parity from {D29*, D30*, 24 data bits << 6}; nib: solve bits 23/24 so that
// D29 = D30 = 0 (words 2 and 10 of a subframe)
uint32_t nav_word(uint32_t source, bool nib) {
    static const uint32_t mask[6] = {0x3B1F3480u, 0x1D8F9A40u, 0x2EC7CD00u, 0x1763E680u, 0x2BB1F340u, 0x0B7A89C0u};
    uint32_t d = source & 0x3FFFFFC0u;
    const unsigned D29 = (source >> 31) & 1u, D30 = (source >> 30) & 1u;
    if (nib) {
        if ((D30 + parity_of(mask[4] & d)) % 2) d ^= (1u << 6);
        if ((D29 + parity_of(mask[5] & d)) % 2) d ^= (1u << 7);
    }
    uint32_t D = d;
    if (D30) D ^= 0x3FFFFFC0u;
    D |= ((D29 + parity_of(mask[0] & d)) % 2) << 5;
    D |= ((D30 + parity_of(mask[1] & d)) % 2) << 4;
    D |= ((D29 + parity_of(mask[2] & d)) % 2) << 3;
    D |= ((D30 + parity_of(mask[3] & d)) % 2) << 2;
    D |= ((D30 + parity_of(mask[4] & d)) % 2) << 1;
    D |= ((D29 + parity_of(mask[5] & d)) % 2);
    D &= 0x3FFFFFFFu;
    D |= (source & 0xC0000000u);
    return D;
}

// ---- SEM almanac reader (almanac.c:73-184) -------------------------------------------------------------------
// The file is read line by line into a 100-byte buffer (fgets), and every record is written in place as it is
// parsed, so a partly read record keeps the fields it got. Layout: "n title", "week sec", then min(n - 1, 31) + 1
// records (unsigned: n = 0 reads 32), each: an optional blank line, ID (0 -> 1, > 32 -> 32; a repeated ID
// overwrites), SVN (may be blank), URA (capped at 15), "e delta_i omegadot", "sqrta omega0 aop", "m0 af0 af1",
// health (capped at 63), config (capped at 15). A complete record gets toa = {week + 2048, sec} and valid = 1.
// A failure before the end of the file drops everything read; a failure at the end of the file keeps it, the
// record it cut short included (svid set, valid 0). Returns -1 when the file cannot be opened, else 0.
int read_sem_almanac(const char *path, Almanac &alm) {
    alm = Almanac();
    FILE *fp = fopen(path, "rt");
    if (!fp) return -1;
    char line[100];
    auto next = [&]() { return fgets(line, sizeof line, fp) != nullptr; };
    auto blank = [&]() { return line[0] == '\n' || line[0] == '\r'; };
    auto parse = [&]() -> bool {
        unsigned n, week, sec, id;
        char title[25];
        if (!next() || sscanf(line, "%u %24s", &n, title) != 2) return false;
        if (!next() || sscanf(line, "%u %u", &week, &sec) != 2) return false;
        const unsigned last = std::min(n - 1u, 31u);
        for (unsigned j = 0; j <= last; j++) {
            if (!next()) return false;
            if (blank() && !next()) return false;
            if (sscanf(line, "%u", &id) != 1) return false;
            id = std::min(std::max(id, 1u), 32u);
            AlmanacSv &a = alm.sv[id - 1];
            a.svid = (unsigned short) id;
            if (!next()) return false;
            if (blank()) a.svn = 0;
            else if (sscanf(line, "%hu", &a.svn) != 1) return false;
            if (!next() || sscanf(line, "%hhu", &a.ura) != 1) return false;
            a.ura = std::min<unsigned char>(a.ura, 15);
            if (!next() || sscanf(line, "%lf %lf %lf", &a.e, &a.delta_i, &a.omegadot) != 3) return false;
            if (!next() || sscanf(line, "%lf %lf %lf", &a.sqrta, &a.omega0, &a.aop) != 3) return false;
            if (!next() || sscanf(line, "%lf %lf %lf", &a.m0, &a.af0, &a.af1) != 3) return false;
            if (!next() || sscanf(line, "%hhu", &a.health) != 1) return false;
            a.health = std::min<unsigned char>(a.health, 63);
            if (!next() || sscanf(line, "%hhu", &a.config_code) != 1) return false;
            a.config_code = std::min<unsigned char>(a.config_code, 15);
            a.toa.week = (int) week + 2048;     // the file's week is modulo 1024 of the current era
            a.toa.sec = (double) sec;
            a.valid = 1;
            alm.valid = 1;
        }
        return true;
    };
    if (!parse() && !feof(fp)) alm = Almanac();
    fclose(fp);
    return 0;
}

// one almanac page (subframe 4 pages 2-5 / 7-10, subframe 5 pages 1-24; gps.c:772-863). toa_scaled is toa.sec / 2^12,
// which the reference spells POW2_12 (an int) in subframe 4 and 4096.0 in subframe 5: the same quotient
void almanac_page(uint32_t w[kWordsPerSbf], unsigned long subframe, int sv, const AlmanacSv &a, double toa_scaled) {
    typedef unsigned long UL;
    const UL dataId = 1, svId = (UL) (sv + 1);
    const UL ecc = (UL) (a.e / P2_21), toa = (UL) toa_scaled, sqrta = (UL) (a.sqrta / P2_11);
    const long delta_i = (long) (a.delta_i / P2_19), omegadot = (long) (a.omegadot / P2_38),
               omega0 = (long) (a.omega0 / P2_23), aop = (long) (a.aop / P2_23), m0 = (long) (a.m0 / P2_23),
               af0 = (long) (a.af0 / P2_20), af1 = (long) (a.af1 / P2_38);
    w[0] = (uint32_t) (0x8B0000UL << 6);
    w[1] = (uint32_t) (subframe << 8);
    w[2] = (uint32_t) ((dataId << 28) | (svId << 22) | ((ecc & 0xFFFFUL) << 6));
    w[3] = (uint32_t) (((toa & 0xFFUL) << 22) | ((delta_i & 0xFFFFUL) << 6));
    w[4] = (uint32_t) ((omegadot & 0xFFFFUL) << 14);            // SV health 0
    w[5] = (uint32_t) ((sqrta & 0xFFFFFFUL) << 6);
    w[6] = (uint32_t) ((omega0 & 0xFFFFFFUL) << 6);
    w[7] = (uint32_t) ((aop & 0xFFFFFFUL) << 6);
    w[8] = (uint32_t) ((m0 & 0xFFFFFFUL) << 6);
    w[9] = (uint32_t) (((af0 & 0x7F8UL) << 19) | ((af1 & 0x7FFUL) << 11) | ((af0 & 0x7UL) << 8));
}

// ---- subframes 1-3 + pages of 4/5 (gps.c:617-884); alm == NULL: the reference with its almanac disabled -----------
void build_subframes(const Eph &e, const IonoUtc &io, const Almanac *alm, uint32_t sbf[kSbfPages][kWordsPerSbf]) {
    typedef unsigned long UL;    // the reference packs in (64-bit) long; only the low 32 bits survive
    const UL wn = 0, ura = 0, dataId = 1, EMPTY = 0xaaaaaaaaUL;
    const UL toe = (UL) (e.toe.sec / 16.0), toc = (UL) (e.toc.sec / 16.0);
    const UL iode = (UL) e.iode, iodc = (UL) e.iodc;
    const long deltan = (long) (e.deltan / P2_43 / kPi);
    const long cuc = (long) (e.cuc / P2_29), cus = (long) (e.cus / P2_29), cic = (long) (e.cic / P2_29),
               cis = (long) (e.cis / P2_29), crc = (long) (e.crc / P2_5), crs = (long) (e.crs / P2_5);
    const UL ecc = (UL) (e.ecc / P2_33), sqrta = (UL) (e.sqrta / P2_19);
    const long m0 = (long) (e.m0 / P2_31 / kPi), omega0 = (long) (e.omg0 / P2_31 / kPi),
               inc0 = (long) (e.inc0 / P2_31 / kPi), aop = (long) (e.aop / P2_31 / kPi),
               omegadot = (long) (e.omgdot / P2_43 / kPi), idot = (long) (e.idot / P2_43 / kPi);
    const long af0 = (long) (e.af0 / P2_31), af1 = (long) (e.af1 / P2_43), af2 = (long) (e.af2 / P2_55),
               tgd = (long) (e.tgd / P2_31);
    const long alpha0 = (long) round(io.alpha[0] / P2_30), alpha1 = (long) round(io.alpha[1] / P2_27),
               alpha2 = (long) round(io.alpha[2] / P2_24), alpha3 = (long) round(io.alpha[3] / P2_24);
    const long beta0 = (long) round(io.beta[0] / 2048.0), beta1 = (long) round(io.beta[1] / 16384.0),
               beta2 = (long) round(io.beta[2] / 65536.0), beta3 = (long) round(io.beta[3] / 65536.0);
    const long A0 = (long) round(io.A0 / P2_30), A1 = (long) round(io.A1 / P2_50);
    const long dtls = (long) io.dtls, dtlsf = 18;
    const UL tot = (UL) (io.tot / 4096), wnt = (UL) (io.wnt % 256), wnlsf = 1929 % 256, dn = 7;
    auto put = [&](int page, int w, UL v) { sbf[page][w] = (uint32_t) v; };
    const UL TLM = 0x8B0000UL << 6;
    put(0, 0, TLM);
    put(0, 1, 0x1UL << 8);
    put(0, 2, ((wn & 0x3FFUL) << 20) | (ura << 14) | (((iodc >> 8) & 0x3UL) << 6));
    put(0, 3, 0);
    put(0, 4, 0);
    put(0, 5, 0);
    put(0, 6, (tgd & 0xFFUL) << 6);
    put(0, 7, ((iodc & 0xFFUL) << 22) | ((toc & 0xFFFFUL) << 6));
    put(0, 8, ((af2 & 0xFFUL) << 22) | ((af1 & 0xFFFFUL) << 6));
    put(0, 9, (af0 & 0x3FFFFFUL) << 8);
    put(1, 0, TLM);
    put(1, 1, 0x2UL << 8);
    put(1, 2, ((iode & 0xFFUL) << 22) | ((crs & 0xFFFFUL) << 6));
    put(1, 3, ((deltan & 0xFFFFUL) << 14) | (((m0 >> 24) & 0xFFUL) << 6));
    put(1, 4, (m0 & 0xFFFFFFUL) << 6);
    put(1, 5, ((cuc & 0xFFFFUL) << 14) | (((ecc >> 24) & 0xFFUL) << 6));
    put(1, 6, (ecc & 0xFFFFFFUL) << 6);
    put(1, 7, ((cus & 0xFFFFUL) << 14) | (((sqrta >> 24) & 0xFFUL) << 6));
    put(1, 8, (sqrta & 0xFFFFFFUL) << 6);
    put(1, 9, (toe & 0xFFFFUL) << 14);
    put(2, 0, TLM);
    put(2, 1, 0x3UL << 8);
    put(2, 2, ((cic & 0xFFFFUL) << 14) | (((omega0 >> 24) & 0xFFUL) << 6));
    put(2, 3, (omega0 & 0xFFFFFFUL) << 6);
    put(2, 4, ((cis & 0xFFFFUL) << 14) | (((inc0 >> 24) & 0xFFUL) << 6));
    put(2, 5, (inc0 & 0xFFFFFFUL) << 6);
    put(2, 6, ((crc & 0xFFFFUL) << 14) | (((aop >> 24) & 0xFFUL) << 6));
    put(2, 7, (aop & 0xFFFFFFUL) << 6);
    put(2, 8, (omegadot & 0xFFFFFFUL) << 6);
    put(2, 9, ((iode & 0xFFUL) << 22) | ((idot & 0x3FFFUL) << 8));
    // subframes 4 and 5: 25 pages each of alternating ones and zeros for the dummy SV
    for (int i = 0; i < 25; i++)
        for (int s = 0; s < 2; s++) {
            const int page = 3 + s + i * 2;
            put(page, 0, TLM);
            put(page, 1, (s == 0 ? 0x4UL : 0x5UL) << 8);
            put(page, 2, (dataId << 28) | (0UL << 22) | ((EMPTY & 0xFFFFUL) << 6));
            for (int w = 3; w < 9; w++) put(page, w, (EMPTY & 0xFFFFFFUL) << 6);
            put(page, 9, (EMPTY & 0x3FFFFFUL) << 8);
        }
    if (alm) {
        // subframe 4 pages 2-5 and 7-10: PRN 25-28 and 29-32, for complete records
        for (int sv = 24; sv < kMaxSat; sv++)
            if (alm->sv[sv].valid != 0) {
                const int i = sv <= 27 ? sv - 23 : sv - 22;
                almanac_page(sbf[3 + i * 2], 0x4UL, sv, alm->sv[sv], alm->sv[sv].toa.sec / P2p12);
            }
        // subframe 5 pages 1-24: PRN 1-24, for every record that was started
        for (int sv = 0; sv < 24; sv++)
            if (alm->sv[sv].svid != 0) almanac_page(sbf[4 + sv * 2], 0x5UL, sv, alm->sv[sv], alm->sv[sv].toa.sec / 4096.0);
    }
    if (io.valid) {                                   // subframe 4 page 18: ionosphere + UTC (SV id 56)
        const int p = 3 + 17 * 2;
        put(p, 0, TLM);
        put(p, 1, 0x4UL << 8);
        put(p, 2, (dataId << 28) | (56UL << 22) | ((alpha0 & 0xFFUL) << 14) | ((alpha1 & 0xFFUL) << 6));
        put(p, 3, ((alpha2 & 0xFFUL) << 22) | ((alpha3 & 0xFFUL) << 14) | ((beta0 & 0xFFUL) << 6));
        put(p, 4, ((beta1 & 0xFFUL) << 22) | ((beta2 & 0xFFUL) << 14) | ((beta3 & 0xFFUL) << 6));
        put(p, 5, (A1 & 0xFFFFFFUL) << 6);
        put(p, 6, ((A0 >> 8) & 0xFFFFFFUL) << 6);
        put(p, 7, ((A0 & 0xFFUL) << 22) | ((tot & 0xFFUL) << 14) | ((wnt & 0xFFUL) << 6));
        put(p, 8, ((dtls & 0xFFUL) << 22) | ((wnlsf & 0xFFUL) << 14) | ((dn & 0xFFUL) << 6));
        put(p, 9, (dtlsf & 0xFFUL) << 22);
    }
    {                                                   // subframe 4 page 25 (SV id 63): health
        const int p = 3 + 24 * 2;
        put(p, 0, TLM);
        put(p, 1, 0x4UL << 8);
        put(p, 2, (dataId << 28) | (63UL << 22));
        for (int w = 3; w < 10; w++) put(p, w, 0);
    }
    {                                                   // subframe 5 page 25 (SV id 51): toa / wna
        const int p = 4 + 24 * 2;
        // of the first started almanac record (its toa stays {0, 0} when it was cut short), else of the ephemeris
        UL wna = (UL) (e.toe.week % 256), toa = (UL) (e.toe.sec / 4096.0);
        for (int sv = 0; alm && sv < kMaxSat; sv++)
            if (alm->sv[sv].svid != 0) {
                wna = (UL) (alm->sv[sv].toa.week % 256);
                toa = (UL) (alm->sv[sv].toa.sec / 4096.0);
                break;
            }
        put(p, 0, TLM);
        put(p, 1, 0x5UL << 8);
        put(p, 2, (dataId << 28) | (51UL << 22) | ((toa & 0xFFUL) << 14) | ((wna & 0xFFUL) << 6));
        for (int w = 3; w < 10; w++) put(p, w, 0);
    }
}

// ---- 30 s NAV frame: previous subframe 5 + subframes 1-5 (gps.c:2066-2140) ---------------------------------
void build_nav_frame(const GpsTime &g, Channel &ch, bool init) {
    GpsTime g0;
    g0.week = g.week;
    g0.sec = (double) (((unsigned long) (g.sec + 0.5)) / 30UL) * 30.0;
    ch.g0 = g0;
    const unsigned long wn = (unsigned long) (g0.week % 1024);
    unsigned long tow = ((unsigned long) g0.sec) / 6UL;
    uint32_t prev = 0;
    if (init) {
        for (int w = 0; w < kWordsPerSbf; w++) {
            uint32_t v = ch.sbf[4 + ch.ipage * 2][w];
            if (w == 1) v |= (uint32_t) ((tow & 0x1FFFFUL) << 13);
            v |= (prev << 30) & 0xC0000000u;
            ch.dwrd[w] = nav_word(v, w == 1 || w == 9);
            prev = ch.dwrd[w];
        }
    } else {
        for (int w = 0; w < kWordsPerSbf; w++) {
            ch.dwrd[w] = ch.dwrd[kWordsPerSbf * 5 + w];
            prev = ch.dwrd[w];
        }
    }
    for (int s = 0; s < 5; s++) {
        tow++;
        for (int w = 0; w < kWordsPerSbf; w++) {
            uint32_t v = s < 3 ? ch.sbf[s][w] : ch.sbf[(s == 3 ? 3 : 4) + ch.ipage * 2][w];
            if (s == 0 && w == 2) v |= (uint32_t) ((wn & 0x3FFUL) << 20);
            if (w == 1) v |= (uint32_t) ((tow & 0x1FFFFUL) << 13);
            v |= (prev << 30) & 0xC0000000u;
            ch.dwrd[(s + 1) * kWordsPerSbf + w] = nav_word(v, w == 1 || w == 9);
            prev = ch.dwrd[(s + 1) * kWordsPerSbf + w];
        }
    }
    if (++ch.ipage >= 25) ch.ipage = 0;
}

// ---- code phase / NAV position at the start of a block (gps.c:2033-2064) -------------------------------------
// A pure function of (the range the reference holds in chan.rho0, the NAV frame start chan.g0, this block's
// range): the form the block-parallel scenario builder needs. Results in `out` (f_carr, f_code, code_phase,
// iword, ibit, icode).
void block_start_pure(const Range &rho0, const GpsTime &frame_g0, const Range &rho1, double dt, gpsb200_chan_t &out) {
    const double rhorate = (rho1.range - rho0.range) / dt;
    out.f_carr = -rhorate / kLambda;
    out.f_code = kCodeFreq + out.f_carr * kCarrToCode;
    const double ms = ((gps_diff(rho0.g, frame_g0) + 6.0) - rho0.range / kC) * 1000.0;
    int ims = (int) ms;
    out.code_phase = (ms - (double) ims) * GPSB200_CA_LEN;
    out.iword = ims / 600;
    ims -= out.iword * 600;
    out.ibit = ims / 20;
    ims -= out.ibit * 20;
    out.icode = ims;
}

// ---- RINEX v2 navigation reader (gps.c:1131-1505) ----------------------------------------------------------------
double field(const std::string &line, size_t pos, size_t len) {
    std::string s = pos < line.size() ? line.substr(pos, len) : std::string();
    for (auto &c : s)
        if (c == 'D' || c == 'd') c = 'E';
    return atof(s.c_str());
}
int ifield(const std::string &line, size_t pos, size_t len) {
    return atoi((pos < line.size() ? line.substr(pos, len) : std::string()).c_str());
}
bool label_is(const std::string &line, const char *label) {
    return line.size() > 60 && line.compare(60, strlen(label), label) == 0;
}

// the seven BROADCAST ORBIT lines of one record; four 19-character fields starting at column c0
// (3 in RINEX 2, 4 in RINEX 3), plus the derived quantities of gps.c:1489-1493
void fill_orbit(Eph &e, const std::string l[7], int c0) {
    e.iode = (int) field(l[0], c0, 19);
    e.crs = field(l[0], c0 + 19, 19);
    e.deltan = field(l[0], c0 + 38, 19);
    e.m0 = field(l[0], c0 + 57, 19);
    e.cuc = field(l[1], c0, 19);
    e.ecc = field(l[1], c0 + 19, 19);
    e.cus = field(l[1], c0 + 38, 19);
    e.sqrta = field(l[1], c0 + 57, 19);
    e.toe.sec = field(l[2], c0, 19);
    e.cic = field(l[2], c0 + 19, 19);
    e.omg0 = field(l[2], c0 + 38, 19);
    e.cis = field(l[2], c0 + 57, 19);
    e.inc0 = field(l[3], c0, 19);
    e.crc = field(l[3], c0 + 19, 19);
    e.aop = field(l[3], c0 + 38, 19);
    e.omgdot = field(l[3], c0 + 57, 19);
    e.idot = field(l[4], c0, 19);
    e.toe.week = (int) field(l[4], c0 + 38, 19);
    e.svh = (int) field(l[5], c0 + 19, 19);
    if (e.svh > 0 && e.svh < 32) e.svh += 32;
    e.tgd = field(l[5], c0 + 38, 19);
    e.iodc = (int) field(l[5], c0 + 57, 19);
    e.valid = true;
    e.A = e.sqrta * e.sqrta;
    e.n = sqrt(kGM / (e.A * e.A * e.A)) + e.deltan;
    e.sq1e2 = sqrt(1.0 - e.ecc * e.ecc);
    e.omgkdot = e.omgdot - kOmegaE;
}

int read_rinex2(const char *path, Eph eph[kEphSets][kMaxSat], IonoUtc &io) {
    gzFile fp = gzopen(path, "rt");                   // plain text or .gz, like the reference (gps.c:1147)
    if (!fp) return -1;
    char buf[256];
    auto next = [&](std::string &out) -> bool {
        if (!gzgets(fp, buf, 100)) return false;      // MAX_CHAR = 100 (gps.h:30)
        out = buf;
        return true;
    };
    std::string ln;
    int flags = 0;
    while (next(ln)) {
        if (label_is(ln, "COMMENT")) continue;
        if (label_is(ln, "END OF HEADER")) break;
        if (label_is(ln, "RINEX VERSION / TYPE")) {
            if (field(ln, 0, 9) > 3.0 || ln.size() <= 20 || ln[20] != 'N') {
                gzclose(fp);
                return -2;
            }
        } else if (label_is(ln, "ION ALPHA")) {
            for (int k = 0; k < 4; k++) io.alpha[k] = field(ln, 2 + 12 * k, 12);
            flags |= 1;
        } else if (label_is(ln, "ION BETA")) {
            for (int k = 0; k < 4; k++) io.beta[k] = field(ln, 2 + 12 * k, 12);
            flags |= 2;
        } else if (label_is(ln, "DELTA-UTC")) {
            io.A0 = field(ln, 3, 19);
            io.A1 = field(ln, 22, 19);
            io.tot = ifield(ln, 41, 9);
            io.wnt = ifield(ln, 50, 9);
            if (io.tot % 4096 == 0) flags |= 4;
        } else if (label_is(ln, "LEAP SECONDS")) {
            io.dtls = ifield(ln, 0, 6);
            flags |= 8;
        }
    }
    io.valid = flags == 0xF;
    GpsTime g0;
    g0.week = -1;
    int ieph = 0;
    while (next(ln)) {
        const int sv = ifield(ln, 0, 2) - 1;
        Date t;
        t.y = ifield(ln, 3, 2) + 2000;
        t.m = ifield(ln, 6, 2);
        t.d = ifield(ln, 9, 2);
        t.hh = ifield(ln, 12, 2);
        t.mm = ifield(ln, 15, 2);
        t.sec = field(ln, 18, 2);                       // the reference keeps two characters of the seconds field
        if (sv < 0 || sv >= kMaxSat || t.m < 1 || t.m > 12) break;
        const GpsTime g = date_to_gps(t);
        if (g0.week == -1) g0 = g;
        if (gps_diff(g, g0) > kSecHour) {
            g0 = g;
            if (++ieph >= kEphSets) break;
        }
        Eph &e = eph[ieph][sv];
        e.t = t;
        e.toc = g;
        e.af0 = field(ln, 22, 19);
        e.af1 = field(ln, 41, 19);
        e.af2 = field(ln, 60, 19);
        std::string l[7];
        bool ok = true;
        for (int k = 0; k < 7 && ok; k++) ok = next(l[k]);
        if (!ok) break;
        fill_orbit(e, l, 3);
    }
    gzclose(fp);
    if (g0.week >= 0) ieph += 1;
    return ieph > kEphSets ? kEphSets : ieph;      // a file with more than 13 hourly sets: the table is full (the
}                                                   // reference returns 14 there and reads past its array)

// ---- RINEX v3 navigation reader (gps.c:1512-1891): GPS records only ------------------------------------------
int read_rinex3(const char *path, Eph eph[kEphSets][kMaxSat], IonoUtc &io) {
    gzFile fp = gzopen(path, "rt");                   // gps.c:1528
    if (!fp) return -1;
    char buf[256];
    auto next = [&](std::string &out) -> bool {
        if (!gzgets(fp, buf, 100)) return false;
        out = buf;
        return true;
    };
    std::string ln;
    int flags = 0;
    while (next(ln)) {
        if (label_is(ln, "COMMENT")) continue;
        if (label_is(ln, "END OF HEADER")) break;
        if (label_is(ln, "RINEX VERSION / TYPE")) {
            if (field(ln, 0, 9) < 3.0 || ln.size() <= 40 || (ln[20] != 'N' && ln[40] != 'G')) {
                gzclose(fp);
                return -2;
            }
        } else if (label_is(ln, "IONOSPHERIC CORR")) {
            if (ln.compare(0, 4, "GPSA") == 0) {
                for (int k = 0; k < 4; k++) io.alpha[k] = field(ln, 5 + 12 * k, 12);
                flags |= 1;
            } else if (ln.compare(0, 4, "GPSB") == 0) {
                for (int k = 0; k < 4; k++) io.beta[k] = field(ln, 5 + 12 * k, 12);
                flags |= 2;
            }
        } else if (label_is(ln, "TIME SYSTEM CORR") && ln.compare(0, 4, "GPUT") == 0) {
            io.A0 = field(ln, 5, 17);
            io.A1 = field(ln, 22, 16);
            io.tot = ifield(ln, 38, 7);
            io.wnt = ifield(ln, 45, 6);
            if (io.tot % 4096 == 0) flags |= 4;
        } else if (label_is(ln, "LEAP SECONDS")) {
            io.dtls = ifield(ln, 0, 6);
            flags |= 8;
        }
    }
    io.valid = flags == 0xF;
    GpsTime g0;
    g0.week = -1;
    int ieph = 0;
    while (next(ln)) {
        if (ln.empty() || ln[0] != 'G') continue;
        const int sv = ifield(ln, 1, 2) - 1;
        Date t;
        t.y = ifield(ln, 4, 4);
        t.m = ifield(ln, 9, 2);
        t.d = ifield(ln, 12, 2);
        t.hh = ifield(ln, 15, 2);
        t.mm = ifield(ln, 18, 2);
        t.sec = (double) ifield(ln, 21, 2);
        if (sv < 0 || sv >= kMaxSat || t.m < 1 || t.m > 12) break;
        const GpsTime g = date_to_gps(t);
        if (g0.week == -1) g0 = g;
        if (gps_diff(g, g0) > kSecHour) {
            g0 = g;
            if (++ieph >= kEphSets) break;
        }
        Eph &e = eph[ieph][sv];
        e.t = t;
        e.toc = g;
        e.af0 = field(ln, 23, 19);
        e.af1 = field(ln, 42, 19);
        e.af2 = field(ln, 61, 19);
        std::string l[7];
        bool ok = true;
        for (int k = 0; k < 7 && ok; k++) ok = next(l[k]);
        if (!ok) break;
        fill_orbit(e, l, 4);
    }
    gzclose(fp);
    if (g0.week >= 0) ieph += 1;
    return ieph;
}

}  // namespace

// =====================================================================================================
struct gpsb200_scenario {
    gpsb200_scenario_config_t cfg{};
    int nchan = 12, nblocks = 0;
    std::vector<gpsb200_chan_t> chans;              // [nblocks][nchan]
    std::vector<uint32_t> nav;                      // [nframes][nchan][60]
    int nframes = 0;
    std::string err;
};

namespace {

int fail(gpsb200_scenario *s, const std::string &m) {
    s->err = m;
    return GPSB200_ERR_ARG;
}

int build(gpsb200_scenario *S) {
    const gpsb200_scenario_config_t &cfg = S->cfg;
    const int C = S->nchan;
    static thread_local Eph eph[kEphSets][kMaxSat];
    for (auto &set : eph)
        for (auto &e : set) e = Eph();
    IonoUtc io;
    io.enable = cfg.ionosphere_enable != 0;
    const int neph = cfg.rinex3 ? read_rinex3(cfg.nav_file, eph, io) : read_rinex2(cfg.nav_file, eph, io);
    if (neph <= 0) return fail(S, "cannot read the RINEX navigation file (wrong version flag, or no ephemeris in it)");

    // receiver positions per 0.1 s (gps.c:2331-2363, 2489-2500)
    int numd = cfg.duration_ds;
    double llh[3] = {cfg.lat_deg / kR2D, cfg.lon_deg / kR2D, cfg.height_m};
    std::vector<double> xyz;
    if (cfg.motion_file && cfg.motion_file[0]) {
        FILE *fp = fopen(cfg.motion_file, "rt");
        if (!fp) return fail(S, "cannot open motion file");
        char str[128];
        while (fgets(str, 100, fp)) {
            double t, x, y, z;
            if (sscanf(str, "%lf,%lf,%lf,%lf", &t, &x, &y, &z) == EOF) break;
            xyz.push_back(x);
            xyz.push_back(y);
            xyz.push_back(z);
        }
        fclose(fp);
        const int got = (int) (xyz.size() / 3);
        if (got <= 0) return fail(S, "empty motion file");
        numd = got > cfg.duration_ds ? cfg.duration_ds : got;
    } else {
        xyz.resize(3);
        llh_to_ecef(llh, xyz.data());
        if (cfg.target_valid) {
            // -t distance,bearing,height: start at a point given relative to the location (gps.c:2348-2357). The CLI
            // stores the bearing in millidegrees (gps-sim.c:148) and the producer divides it back: same round trip here.
            double t[3][3], neu[3];
            local_frame(llh, t);
            const double bearing_milli = cfg.target_bearing_deg * 1000;
            neu[0] = cfg.target_distance_m * cos((bearing_milli / 1000) / kR2D);
            neu[1] = cfg.target_distance_m * sin((bearing_milli / 1000) / kR2D);
            neu[2] = cfg.target_height_m;
            xyz[0] += t[0][0] * neu[0] + t[1][0] * neu[1] + t[2][0] * neu[2];
            xyz[1] += t[0][1] * neu[0] + t[1][1] * neu[1] + t[2][1] * neu[2];
            xyz[2] += t[0][2] * neu[0] + t[1][2] * neu[1] + t[2][2] * neu[2];
        }
    }
    auto pos_at = [&](int i) -> const double * { return xyz.size() > 3 ? &xyz[3 * (size_t) i] : xyz.data(); };
    if (numd < 2) return fail(S, "duration too short");

    // scenario start (gps.c:2502-2577)
    GpsTime gmin, gmax, g0;
    bool have = false;
    for (int sv = 0; sv < kMaxSat && !have; sv++)
        if (eph[0][sv].valid) {
            gmin = eph[0][sv].toc;
            have = true;
        }
    for (int sv = 0; sv < kMaxSat; sv++)
        if (eph[neph - 1][sv].valid) {
            gmax = eph[neph - 1][sv].toc;
            break;
        }
    if (cfg.start_year > 0) {
        Date t;
        t.y = cfg.start_year;
        t.m = cfg.start_month;
        t.d = cfg.start_day;
        t.hh = cfg.start_hour;
        t.mm = cfg.start_min;
        t.sec = cfg.start_sec;
        if (t.m < 1 || t.m > 12) return fail(S, "invalid start date");
        g0 = date_to_gps(t);
        if (gps_diff(g0, gmin) < 0.0 || gps_diff(gmax, g0) < 0.0) return fail(S, "start time outside the ephemeris span");
    } else {
        g0 = gmin;
    }
    int ieph = -1;
    for (int i = 0; i < neph && ieph < 0; i++)
        for (int sv = 0; sv < kMaxSat; sv++)
            if (eph[i][sv].valid) {
                const double dt = gps_diff(g0, eph[i][sv].toc);
                if (dt >= -kSecHour && dt < kSecHour) {
                    ieph = i;
                    break;
                }
            }
    if (ieph < 0) return fail(S, "no current set of ephemerides");

    // almanac (gps.c:2614-2651): an unreadable file is the caller's error; a malformed one is read as the
    // reference reads it. A complete record whose toa is more than 4 weeks from the start stops the reference
    // before its first block.
    Almanac alm;
    const bool use_alm = cfg.almanac_file != nullptr;
    if (use_alm) {
        if (read_sem_almanac(cfg.almanac_file, alm) != 0) return fail(S, std::string("cannot open almanac file ") + cfg.almanac_file);
        if (alm.valid)
            for (int sv = 0; sv < kMaxSat; sv++)
                if (alm.sv[sv].valid != 0) {
                    const double dt = gps_diff(alm.sv[sv].toa, g0);
                    if (dt < -4.0 * kSecWeek || dt > 4.0 * kSecWeek)
                        return fail(S, "invalid time of almanac: the toa of PRN " + std::to_string(sv + 1) +
                                           " is more than 4 weeks from the start time");
                }
    }
    const Almanac *almp = use_alm ? &alm : nullptr;

    std::vector<Channel> chan(C);
    std::vector<char> fresh(C, 0);                  // slot (re)allocated since the last epoch snapshot
    int allocated[kMaxSat];
    for (int sv = 0; sv < kMaxSat; sv++) allocated[sv] = -1;
    double ant_pat[37];
    for (int i = 0; i < 37; i++) ant_pat[i] = pow(10.0, -kAntPatDb[i] / 20.0);

    // visibility + channel allocation (gps.c:2142-2235); always evaluated at the INITIAL position
    auto allocate = [&](const Eph *set, const GpsTime &grx) {
        const double *p0 = pos_at(0);
        double llh0[3], tm[3][3];
        ecef_to_llh(p0, llh0);
        local_frame(llh0, tm);
        for (int sv = 0; sv < kMaxSat; sv++) {
            bool visible = false;
            double az = 0, el = 0;
            if (set[sv].valid) {
                double pos[3], vel[3], clk[2], los[3];
                sat_state(set[sv], grx, pos, vel, clk);
                for (int k = 0; k < 3; k++) los[k] = pos[k] - p0[k];
                az_el(los, tm, az, el);
                visible = el * kR2D > 0.0;
            }
            if (visible) {
                if (allocated[sv] == -1) {
                    int i = 0;
                    for (; i < C; i++)
                        if (chan[i].prn == 0) {
                            Channel &ch = chan[i];
                            ch.prn = sv + 1;
                            fresh[i] = 1;
                            // the reference never initialises channel_t.ipage (gps.c:2086 reads it);
                            // its -Og build sees zeroed stack there, which is what is reproduced here
                            build_subframes(set[sv], io, almp, ch.sbf);
                            build_nav_frame(grx, ch, true);
                            const Range r = pseudo_range(set[sv], io, grx, p0);
                            ch.rho0 = r;
                            const double ref[3] = {0.0, 0.0, 0.0};
                            const Range rr = pseudo_range(set[sv], io, grx, ref);
                            const double phase_ini = (2.0 * rr.range - r.range) / kLambda;
                            ch.carr_phase = phase_ini - floor(phase_ini);
                            // integer carrier build (gps.c:2212-2213): the same fraction as a u32 accumulator
                            if (cfg.carrier_u32) ch.carr_phase = (double) (unsigned int) (512.0 * 65536.0 * ch.carr_phase);
                            break;
                        }
                    if (i < C) allocated[sv] = i;
                }
            } else if (allocated[sv] >= 0) {
                chan[allocated[sv]].prn = 0;
                allocated[sv] = -1;
            }
        }
    };

    // The reference's loop (gps.c:2731-2930) does two things per 0.1 s block: the per-channel range /
    // code-phase / gain update, which depends only on this block's and the previous block's range, and,
    // every 30 s, the NAV frame roll / ephemeris roll / reallocation. Here: (A) one cheap sequential pass
    // runs the 30 s events and records, per EPOCH (the blocks between two events), which satellite sits in
    // which slot, with which ephemeris set and NAV frame; (B) all ranges and (C) all block-start states are
    // then computed block-parallel. Every number comes out of the same function with the same arguments
    // as in the sequential order, so the result is bit-identical (tests/test_scenario.py).
    struct Epoch {
        int b_first = 0, ieph = 0;
        std::vector<int> prn;
        std::vector<char> fresh;
        std::vector<GpsTime> frame_g0;
        std::vector<Range> rho_alloc;
        std::vector<double> carr_phase;
    };
    std::vector<Epoch> epochs;
    auto snapshot = [&](int b_first, int ieph_now) {
        Epoch e;
        e.b_first = b_first;
        e.ieph = ieph_now;
        e.prn.resize(C);
        e.fresh = fresh;
        e.frame_g0.resize(C);
        e.rho_alloc.resize(C);
        e.carr_phase.resize(C);
        for (int i = 0; i < C; i++) {
            e.prn[i] = chan[i].prn;
            e.frame_g0[i] = chan[i].g0;
            e.rho_alloc[i] = chan[i].rho0;           // only read where fresh[i]
            e.carr_phase[i] = chan[i].carr_phase;
        }
        std::fill(fresh.begin(), fresh.end(), 0);
        epochs.push_back(std::move(e));
    };

    GpsTime grx = gps_add(g0, 0.0);
    allocate(eph[ieph], grx);
    grx = gps_add(grx, 0.1);

    S->nblocks = numd - 1;
    const int NB = S->nblocks;
    S->chans.assign((size_t) NB * C, gpsb200_chan_t{});
    S->nav.clear();
    S->nframes = 0;
    std::vector<GpsTime> grx_of(NB);
    std::vector<int> epoch_of(NB), frame_of(NB);
    std::vector<uint32_t> cur((size_t) C * GPSB200_NAV_WORDS, 0), last;
    // ---- (A) sequential: times, 30 s events, NAV frame table ------------------------------------------------
    snapshot(0, ieph);
    bool words_may_have_changed = true;
    for (int iumd = 1; iumd < numd; iumd++) {
        const int b = iumd - 1;
        grx_of[b] = grx;
        epoch_of[b] = (int) epochs.size() - 1;
        // NAV frame table: a new frame whenever any channel's words changed (every 30 s / reallocation)
        if (words_may_have_changed) {
            for (int i = 0; i < C; i++)
                for (int k = 0; k < GPSB200_NAV_WORDS; k++)
                    cur[(size_t) i * GPSB200_NAV_WORDS + k] = chan[i].prn > 0 ? chan[i].dwrd[k] : 0u;
            if (cur != last) {
                S->nav.insert(S->nav.end(), cur.begin(), cur.end());
                S->nframes++;
                last = cur;
            }
            words_may_have_changed = false;
        }
        frame_of[b] = S->nframes - 1;
        // every 30 s: NAV frame roll, ephemeris set roll, reallocation (gps.c:2870-2930)
        const int igrx = (int) (grx.sec * 10.0 + 0.5);
        if (igrx % 300 == 0) {
            for (int i = 0; i < C; i++)
                if (chan[i].prn > 0) build_nav_frame(grx, chan[i], false);
            if (ieph + 1 < kEphSets)
                for (int sv = 0; sv < kMaxSat; sv++)
                    if (eph[ieph + 1][sv].valid) {
                        if (gps_diff(eph[ieph + 1][sv].toc, grx) < kSecHour) {
                            ieph++;
                            for (int i = 0; i < C; i++)
                                if (chan[i].prn != 0) build_subframes(eph[ieph][chan[i].prn - 1], io, almp, chan[i].sbf);
                        }
                        break;
                    }
            allocate(eph[ieph], grx);
            if (iumd + 1 < numd) snapshot(b + 1, ieph);
            words_may_have_changed = true;
        }
        grx = gps_add(grx, 0.1);
    }

    // ---- (B) + (C) block-parallel ----------------------------------------------------------------------------
    const Eph(*E)[kMaxSat] = eph;                   // `eph` is thread_local: hand the workers THIS thread's table
    std::vector<Range> rho((size_t) NB * C);
    int nthr = (int) std::thread::hardware_concurrency();
    if (const char *ev = getenv("GPSB200_SCENARIO_THREADS")) nthr = atoi(ev);
    nthr = std::max(1, std::min(std::min(nthr, 16), NB / 64 + 1));
    auto parallel_blocks = [&](const std::function<void(int, int)> &job) {
        if (nthr == 1) {
            job(0, NB);
            return;
        }
        std::vector<std::thread> th;
        const int per = (NB + nthr - 1) / nthr;
        for (int t = 0; t < nthr; t++) {
            const int lo = t * per, hi = std::min(NB, lo + per);
            if (lo < hi) th.emplace_back(job, lo, hi);
        }
        for (auto &t : th) t.join();
    };
    parallel_blocks([&](int lo, int hi) {            // (B) this block's pseudorange per channel (gps.c:2738)
        for (int b = lo; b < hi; b++) {
            const Epoch &ep = epochs[epoch_of[b]];
            for (int i = 0; i < C; i++)
                if (ep.prn[i] > 0) rho[(size_t) b * C + i] = pseudo_range(E[ep.ieph][ep.prn[i] - 1], io, grx_of[b], pos_at(b + 1));
        }
    });
    parallel_blocks([&](int lo, int hi) {            // (C) block-start state and gain (gps.c:2744-2763)
        for (int b = lo; b < hi; b++) {
            const Epoch &ep = epochs[epoch_of[b]];
            for (int i = 0; i < C; i++) {
                gpsb200_chan_t &o = S->chans[(size_t) b * C + i];
                o.nav_frame = frame_of[b];
                if (ep.prn[i] <= 0) continue;
                const Range &r1 = rho[(size_t) b * C + i];
                // the range the reference still holds in chan[i].rho0: the allocation's for a slot's first
                // block, else the previous block's (possibly computed with the previous ephemeris set)
                const Range &r0 = (b == ep.b_first && ep.fresh[i]) ? ep.rho_alloc[i] : rho[(size_t) (b - 1) * C + i];
                block_start_pure(r0, ep.frame_g0[i], r1, 0.1, o);
                const double path_loss = 20200000.0 / r1.d;                     // gps.c:2749
                const int ibs = (int) ((90.0 - r1.el * kR2D) / 5.0);
                double gain = (double) (path_loss * ant_pat[ibs]);
                if (cfg.pluto_gain) gain *= 2;                                  // gps.c:2759-2763
                o.prn = ep.prn[i];
                o.carr_phase = ep.carr_phase[i];   // meaningful for a slot's first block only
                o.gain = gain;
            }
        }
    });
    return GPSB200_OK;
}

}  // namespace

extern "C" {

int gpsb200_scenario_create(const gpsb200_scenario_config_t *cfg, gpsb200_scenario_t **out) {
    if (!cfg || !out || !cfg->nav_file) return GPSB200_ERR_ARG;
    gpsb200_scenario *S = new gpsb200_scenario();
    S->cfg = *cfg;
    S->nchan = cfg->max_chan > 0 ? cfg->max_chan : 12;
    *out = S;
    if (S->nchan > GPSB200_MAX_CHAN) return fail(S, "max_chan > 32");
    return build(S);
}

void gpsb200_scenario_destroy(gpsb200_scenario_t *s) { delete s; }

const char *gpsb200_scenario_error(const gpsb200_scenario_t *s) { return s ? s->err.c_str() : "null scenario"; }

int gpsb200_scenario_blocks(const gpsb200_scenario_t *s) { return s ? s->nblocks : 0; }
int gpsb200_scenario_channels(const gpsb200_scenario_t *s) { return s ? s->nchan : 0; }
int gpsb200_scenario_nav_frames(const gpsb200_scenario_t *s) { return s ? s->nframes : 0; }
const gpsb200_chan_t *gpsb200_scenario_chans(const gpsb200_scenario_t *s) { return s ? s->chans.data() : nullptr; }
const uint32_t *gpsb200_scenario_nav(const gpsb200_scenario_t *s) { return s ? s->nav.data() : nullptr; }

}  // extern "C"
