#!/usr/bin/env python3
"""TEST INFRASTRUCTURE -- deterministic SEM almanac files for the sky-N constellations of gen_rinex.py.

The records are those of the sky-32 constellation (sky-N for N < 32 is its first N satellites), in SEM units:
angles in semicircles, inclination as an offset from 0.30 semicircles, rates in semicircles/s. Some of the signs are
flipped so that every signed field (delta_i, omegadot, omega0, aop, m0, af0, af1) is negative in some record. The
records of PRN 1, 5, 9, ... 29 put every field a few ulps below an exact multiple of its scale factor (2^-21, 2^-19,
2^-38, 2^-11, 2^-23, 2^-20): the reference divides by the literals of gps.h:79-84, two of which (POW2_M38, POW2_M23)
are a little smaller than the true powers of two, so a reader that divides by true powers of two packs different
words there. No RNG anywhere.

--case writes one of the edge-case files the reference's reader (almanac.c:73-184) treats specially:
  ids        ID 0 (read as 1), ID 40 (read as 32), and ID 2 twice (the second record wins)
  short      10 records announced, 3 in the file (kept: the read fails at the end of the file)
  truncated  PRN 25 complete, then PRN 2 cut off in its "sqrta omega0 aop" line at the end of the file
             (kept with the fields read so far, not valid)
  badline    a malformed URA line in the middle of the file (everything is dropped)
  blank      blank SVN lines and blank separator lines, one of them CR LF
  count0     header count 0 (unsigned wrap: up to 32 records are read) with 3 records
Usage: gen_almanac.py --out almanac.sem [--case NAME] [--week W] [--toa S]
"""
import argparse
import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gen_rinex  # noqa: E402

WEEK = gen_rinex.WEEK - 2048      # the SEM file's week: the reader adds 2048
TOA = 15 * 4096                   # 61440 s into the week, a multiple of 2^12 as broadcast
TITLE = "GPSB200.ALM"             # the reference scans it with %24s into a 24-byte buffer: keep it <= 23 characters

# scale factor of each field as an exact power of two
SCALE = {"e": 2.0 ** -21, "delta_i": 2.0 ** -19, "omegadot": 2.0 ** -38, "sqrta": 2.0 ** -11, "omega0": 2.0 ** -23,
         "aop": 2.0 ** -23, "m0": 2.0 ** -23, "af0": 2.0 ** -20, "af1": 2.0 ** -38}


def below_multiple(v, scale, ulps=3):
    """A value `ulps` ulps closer to zero than the nearest nonzero multiple of scale, with the sign of v."""
    k = max(1, int(round(abs(v) / scale)))
    x = k * scale
    for _ in range(ulps):
        x = math.nextafter(x, 0.0)
    return math.copysign(x, v) if v != 0 else x


def records():
    """PRN -> dict of the SEM fields, for PRN 1..32."""
    out = {}
    for prn, (lat, lon) in zip(range(1, 33), gen_rinex.sub_points(32)):
        el = gen_rinex.elements(prn, lat, lon)
        r = dict(
            svn=prn + 40, ura=prn % 3,
            e=el["ecc"],
            delta_i=el["inc"] / math.pi - 0.30 - (0.012 if prn % 2 else 0.0),
            omegadot=(1 if prn % 3 == 0 else -1) * 8e-9 / math.pi,
            sqrta=el["sqrta"],
            omega0=el["omg0"] / math.pi,
            aop=(-1 if prn % 2 else 1) * 0.01 * prn / 32,
            m0=el["m0"] / math.pi,
            af0=(-1 if prn % 2 == 0 else 1) * 1e-5 * prn,
            af1=(-1 if prn % 3 == 1 else 1) * 1e-12 * prn,
            health=0, config=9 + prn % 3)
        if prn % 4 == 1:
            for f, s in SCALE.items():
                r[f] = below_multiple(r[f], s)
        out[prn] = r
    return out


def num(v):
    return "% .16E" % v


def record_lines(id_, r, svn_blank=False):
    """The eight lines of one record, without the separator."""
    return ["%d" % id_, "" if svn_blank else "%d" % r["svn"], "%d" % r["ura"],
            " ".join(num(r[f]) for f in ("e", "delta_i", "omegadot")),
            " ".join(num(r[f]) for f in ("sqrta", "omega0", "aop")),
            " ".join(num(r[f]) for f in ("m0", "af0", "af1")),
            "%d" % r["health"], "%d" % r["config"]]


def text(case=None, week=WEEK, toa=TOA):
    R = records()
    head = lambda n: ["%d %s" % (n, TITLE), " %d %d" % (week, toa)]   # noqa: E731

    def body(entries):
        """entries: (id, prn of the data, svn blank) -> lines with a blank separator before each record"""
        L = []
        for id_, prn, svn_blank in entries:
            L += [""] + record_lines(id_, R[prn], svn_blank)
        return L

    if case is None:
        L = head(32) + body([(p, p, False) for p in range(1, 33)])
    elif case == "ids":
        L = head(5) + body([(0, 1, False), (2, 3, False), (25, 25, False), (2, 2, False), (40, 32, False)])
    elif case == "short":
        L = head(10) + body([(2, 2, False), (25, 25, False), (1, 1, False)])
    elif case == "truncated":
        L = head(3) + body([(25, 25, False), (2, 2, False)])
        L = L[:-4] + [num(R[2]["sqrta"]) + " " + num(R[2]["omega0"])]   # ends mid-line, no newline
        return "\n".join(L)
    elif case == "badline":
        L = head(3) + body([(1, 1, False), (2, 2, False), (25, 25, False)])
        L[2 + 9 + 3] = "x"                                               # URA line of the second record
    elif case == "blank":
        L = head(3) + body([(1, 1, True), (2, 2, False), (25, 25, True)])
        L[2 + 9] = "\r"                                                  # CR LF separator before the second record
    elif case == "count0":
        L = head(0) + body([(1, 1, False), (25, 25, False), (2, 2, False)])
    else:
        raise SystemExit("unknown case %r" % case)
    return "\n".join(L) + "\n"


CASES = ["ids", "short", "truncated", "badline", "blank", "count0"]

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--case", choices=CASES)
    ap.add_argument("--week", type=int, default=WEEK, help="week of the header line (the reader adds 2048)")
    ap.add_argument("--toa", type=int, default=TOA)
    a = ap.parse_args()
    with open(a.out, "w", newline="") as f:
        f.write(text(a.case, a.week, a.toa))
