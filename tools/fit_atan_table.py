#!/usr/bin/env python
"""Prints the arctangent table and series of pm_math.cuh's atan_ratio (paste over the kAtanT / kAtanC
definitions there):   python tools/fit_atan_table.py

atan_ratio reduces q = mn / mx in [0, 1] about the nearest tabulated point t0 = k / 2^M:
    atan(q) = atan(t0) + atan(r),   r = (mn - t0 mx) / (mx + t0 mn).
k comes from a ~20-bit reciprocal seed, so it can be off by one: |r| <= 2^-M covers that with room
to spare (the exact index gives |r| <= 2^-(M+1)).  Over |r| <= 2^-M the Taylor series
atan(r) = r + r z (-1/3 + z/5 - z^2/7),  z = r^2,  leaves r^9 / 9, i.e. < 2^-67 relative to r (checked
below), far under the rounding of the result: the Taylor coefficients need no minimax fit.
Each entry is (t0, atan(t0)) rounded to nearest from 60-digit values, read as one 16-byte load.
"""
import mpmath as mp

M = 8
N = (1 << M) + 1   # k = 0 .. 2^M (q = 1 included)
mp.mp.dps = 60


def series_check():
    lim = mp.mpf(2) ** -M
    c = [mp.mpf(-1) / 3, mp.mpf(1) / 5, mp.mpf(-1) / 7]
    worst = mp.mpf(0)
    for i in range(1, 2001):
        r = lim * i / 2000
        z = r * r
        approx = r + r * z * (c[0] + z * (c[1] + z * c[2]))
        worst = max(worst, abs(approx / mp.atan(r) - 1))
    return worst


def main():
    err = series_check()
    assert err < mp.mpf(2) ** -67, err
    print('// atan(r) = r + r z (c1 + c2 z + c3 z^2), |r| <= 2^-%d: relative truncation error %s' % (M, mp.nstr(err, 3)))
    print('PM_DEV_TABLE(kAtanC, 3, %s, %s, %s)' % tuple(repr(float(mp.mpf(n) / d)) for n, d in ((-1, 3), (1, 5), (-1, 7))))
    vals = []
    for k in range(N):
        t0 = mp.mpf(k) / (1 << M)
        vals.append('%s, %s' % (repr(float(t0)), repr(float(mp.atan(t0)))))
    print('// (k / 2^%d, atan(k / 2^%d)) for k = 0 .. %d' % (M, M, N - 1))
    print('PM_LDG_TABLE(kAtanT, %d,' % (2 * N))
    print(',\n'.join('             ' + v for v in vals) + ')')


if __name__ == '__main__':
    main()
