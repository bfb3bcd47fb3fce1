// pm_regrid.cuh - FITPACK's smoothing spline on a rectangular grid (regrid / fpregr, iopt = 0), the
// fit behind RectBivariateSpline(x, y, z, kx, ky, s > 0), written once for the host and the device.
//
// The control flow (knot growth, then the iteration on the smoothing parameter p) is a restatement of
// fpregr; the least-squares step is fpgrre with the banded Givens QR split into a scalar part (the
// rotation parameters of one row, one thread) and a per-column part (the rotated right-hand sides, one
// thread per column).  Every scalar is computed by exactly one thread and every sum is taken in
// FITPACK's loop order, so the knot decisions (|fp - s| < acc, fpmax >= fpint(j), int(rn fpms / reduc))
// come out as FITPACK's, and the host and device builds agree bit for bit.  Division and square root
// are IEEE (correctly rounded) on both sides; the file is compiled without FMA contraction.
//
// Grid and coefficient conventions (FITPACK's names): "x" is the slow axis of z (mx points, degree kx),
// "y" the fast axis (my points, degree ky); the data sites are x = 0 .. mx-1, y = 0 .. my-1 (np.arange)
// and the bounding box is their range.  c[i * (ny - ky - 1) + j] multiplies B_i(x) B_j(y).
#pragma once

#include <cmath>
#include <cstdint>

#if defined(__CUDACC__)
#define PMR_HD __host__ __device__
#else
#define PMR_HD
#endif

namespace pm {
namespace regrid {

PMR_HD inline double div_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
PMR_HD inline double sqrt_rn(double a) {
#if defined(__CUDA_ARCH__)
    return __dsqrt_rn(a);
#else
    return std::sqrt(a);
#endif
}
// Fortran / C double -> integer conversion as the x86-64 build of FITPACK performs it (cvttsd2si):
// truncation, and INT_MIN for NaN or out-of-range values (the device instruction would saturate).
PMR_HD inline int trunc_to_int(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return (int)0x80000000u;
    return (int)v;
}

constexpr int kMaxK = 3;             // degrees 1..3 per axis
constexpr double kTol = 0.001;       // regrid's tol: acc = tol * s
constexpr double kCon1 = 0.1, kCon4 = 0.04, kCon9 = 0.9;

// scipy's ier values that come out of the fit
enum : int { kIerLsqPoly = -2, kIerInterp = -1, kIerOk = 0, kIerNest = 1, kIerTheory = 2, kIerMaxit = 3,
             kIerInput = 10 };

// Per-plane workspace (doubles then ints), sized by work_doubles / work_ints.
struct Work {
    double *spx, *spy;      // [mx][kx+1], [my][ky+1] non-zero B-spline values at the data sites
    double *q;              // [nxest - kx - 1][my]: x-rotated right-hand sides
    double *ax, *bx;        // [nxest][kx+2] triangle / penalty rows along x
    double *ay, *by;        // [nyest][ky+2]
    double *term;           // [mx][my] squared residuals
    double *fpintx, *fpinty;// [nxest], [nyest]
    int *nrx, *nry;         // [mx], [my] knot interval of each data site
    int *nrdatx, *nrdaty;   // [nxest], [nyest] interior data sites per knot interval
};
PMR_HD inline int64_t work_doubles(int mx, int my, int kx, int ky, int nxest, int nyest) {
    return (int64_t)mx * (kx + 1) + (int64_t)my * (ky + 1) + (int64_t)(nxest - kx - 1) * my +
           2 * (int64_t)nxest * (kx + 2) + 2 * (int64_t)nyest * (ky + 2) + (int64_t)mx * my + nxest + nyest;
}
PMR_HD inline int64_t work_ints(int mx, int my, int nxest, int nyest) {
    return (int64_t)mx + my + nxest + nyest;
}
PMR_HD inline Work carve(double *d, int *iw, int mx, int my, int kx, int ky, int nxest, int nyest) {
    Work w;
    w.spx = d; d += (int64_t)mx * (kx + 1);
    w.spy = d; d += (int64_t)my * (ky + 1);
    w.q = d; d += (int64_t)(nxest - kx - 1) * my;
    w.ax = d; d += (int64_t)nxest * (kx + 2);
    w.bx = d; d += (int64_t)nxest * (kx + 2);
    w.ay = d; d += (int64_t)nyest * (ky + 2);
    w.by = d; d += (int64_t)nyest * (ky + 2);
    w.term = d; d += (int64_t)mx * my;
    w.fpintx = d; d += nxest;
    w.fpinty = d;
    w.nrx = iw; iw += mx;
    w.nry = iw; iw += my;
    w.nrdatx = iw; iw += nxest;
    w.nrdaty = iw;
    return w;
}

// ---- FITPACK's scalar kernels (fpgivs, fprota, fpbspl, fpback, fpdisc, fprati) ----------------------
PMR_HD inline void fpgivs(double piv, double &ww, double &cos, double &sin) {
    const double store = fabs(piv);
    double dd;
    if (store >= ww) {
        const double r = div_rn(ww, piv);
        dd = store * sqrt_rn(1.0 + r * r);
    } else {
        const double r = div_rn(piv, ww);
        dd = ww * sqrt_rn(1.0 + r * r);
    }
    cos = div_rn(ww, dd);
    sin = div_rn(piv, dd);
    ww = dd;
}
PMR_HD inline void fprota(double cos, double sin, double &a, double &b) {
    const double stor1 = a, stor2 = b;
    b = cos * stor2 + sin * stor1;
    a = cos * stor1 - sin * stor2;
}
// The k+1 non-zero B-splines of degree k at x, t(l) <= x < t(l+1); t and l are 1-based as in FITPACK
// (t1[i] = t(i)), h[0..k].
PMR_HD inline void fpbspl(const double *t1, int k, double x, int l, double *h) {
    double hh[kMaxK + 1];
    h[0] = 1.0;
    for (int j = 1; j <= k; j++) {
        for (int i = 0; i < j; i++) hh[i] = h[i];
        h[0] = 0.0;
        for (int i = 1; i <= j; i++) {
            const int li = l + i, lj = li - j;
            if (t1[li] == t1[lj]) {
                h[i] = 0.0;
                continue;
            }
            const double f = div_rn(hh[i - 1], t1[li] - t1[lj]);
            h[i - 1] = h[i - 1] + f * (t1[li] - x);
            h[i] = f * (x - t1[lj]);
        }
    }
}
// Solve a c = z in place (c = z) for the n x n upper triangular band matrix a[row][0..k-1] (row stride
// lda); element i of c is c[i * stride].
PMR_HD inline void fpback_inplace(const double *a, int lda, double *c, int64_t stride, int n, int k) {
    const int k1 = k - 1;
    c[(int64_t)(n - 1) * stride] = div_rn(c[(int64_t)(n - 1) * stride], a[(int64_t)(n - 1) * lda]);
    int i = n - 2;
    for (int j = 2; j <= n; j++, i--) {
        double store = c[(int64_t)i * stride];
        const int i1 = j <= k1 ? j - 1 : k1;
        int m = i;
        for (int l = 1; l <= i1; l++) {
            m++;
            store = store - c[(int64_t)m * stride] * a[(int64_t)i * lda + l];
        }
        c[(int64_t)i * stride] = div_rn(store, a[(int64_t)i * lda]);
    }
}
// Row lmk (0-based) of the discontinuity-jump matrix of the k-th derivative (fpdisc), k2 = k + 2.
PMR_HD inline void fpdisc_row(const double *t1, int n, int k2, int lmk, double *b) {
    const int k1 = k2 - 1, k = k1 - 1, nk1 = n - k1, nrint = nk1 - k;
    const double an = nrint;
    const double fac = div_rn(an, t1[nk1 + 1] - t1[k1]);
    const int l = lmk + 1 + k1;
    double h[2 * (kMaxK + 1)];
    for (int j = 1; j <= k1; j++) {
        const int lj = l + j, lk = lj - k2;
        h[j - 1] = t1[l] - t1[lk];
        h[j + k1 - 1] = t1[l] - t1[lj];
    }
    int lp = lmk + 1;
    for (int j = 1; j <= k2; j++) {
        int jk = j;
        double prod = h[j - 1];
        for (int i = 1; i <= k; i++) {
            jk++;
            prod = prod * h[jk - 1] * fac;
        }
        const int lk = lp + k1;
        b[j - 1] = div_rn(t1[lk] - t1[lp], prod);
        lp++;
    }
}
PMR_HD inline double fprati(double &p1, double &f1, double p2, double f2, double &p3, double &f3) {
    double p;
    if (!(p3 > 0.0)) {
        p = div_rn(p1 * (f1 - f3) * f2 - p2 * (f2 - f3) * f1, (f1 - f2) * f3);
    } else {
        const double h1 = f1 * (f2 - f3), h2 = f2 * (f3 - f1), h3 = f3 * (f1 - f2);
        p = -div_rn(p1 * p2 * h3 + p2 * p3 * h1 + p3 * p1 * h2, p1 * h1 + p2 * h2 + p3 * h3);
    }
    if (f2 < 0.0) {
        p3 = p2;
        f3 = f2;
    } else {
        p1 = p2;
        f1 = f2;
    }
    return p;
}
// Knot interval of x (fpbisp / fpgrre search, 1-based): the smallest l in [k+1, n-k-1] with
// x < t(l+1), or n-k-1.
PMR_HD inline int knot_interval(const double *t1, int n, int k, double x) {
    int lo = k + 1, hi = n - k - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (x < t1[mid + 1]) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}
// fpknot with istart = 1 and data sites x(i) = i - 1: one knot in the interval of largest fpint among
// those with interior data sites, at its middle data site; fpint / nrdata split in proportion.
// Arrays are 1-based views (fpint1[j] = fpint(j)).
PMR_HD inline void fpknot(double *t1, int &n, double *fpint1, int *nrdata1, int &nrint) {
    const int k = (n - nrint - 1) / 2;
    double fpmax = 0.0;
    int jbegin = 1, number = 1, maxpt = 0, maxbeg = 1;
    for (int j = 1; j <= nrint; j++) {
        const int jpoint = nrdata1[j];
        if (!(fpmax >= fpint1[j] || jpoint == 0)) {
            fpmax = fpint1[j];
            number = j;
            maxpt = jpoint;
            maxbeg = jbegin;
        }
        jbegin = jbegin + jpoint + 1;
    }
    const int ihalf = maxpt / 2 + 1;
    const int nrx = maxbeg + ihalf;
    const int next = number + 1;
    for (int j = next; j <= nrint; j++) {
        const int jj = next + nrint - j;
        fpint1[jj + 1] = fpint1[jj];
        nrdata1[jj + 1] = nrdata1[jj];
        const int jk = jj + k;
        t1[jk + 1] = t1[jk];
    }
    nrdata1[number] = ihalf - 1;
    nrdata1[next] = maxpt - ihalf;
    const double am = maxpt;
    double an = nrdata1[number];
    fpint1[number] = div_rn(fpmax * an, am);
    an = nrdata1[next];
    fpint1[next] = div_rn(fpmax * an, am);
    t1[next + k] = (double)(nrx - 1);
    n = n + 1;
    nrint = nrint + 1;
}

// Interior knots of the interpolating spline (fpregr's s = 0 branch) for data sites x(i) = i - 1:
// the sites themselves for odd k, the midpoints for even k.  t1 is 1-based.
PMR_HD inline void interpolation_knots(double *t1, int m, int k) {
    const int k3 = k / 2;
    for (int l = 1, i = k + 2, j = k3 + 2; l <= m - k - 1; l++, i++, j++)
        t1[i] = (k3 * 2 == k) ? ((double)(j - 1) + (double)(j - 2)) * 0.5 : (double)(j - 1);
}

// ---- fpregr's control state ------------------------------------------------------------------------
struct Ctl {
    int mx, my, kx, ky, nxest, nyest, maxit;
    double s, acc;
    int nx, ny, nminx, nminy, nmaxx, nmaxy, nxe, nye, nrintx, nrinty;
    int lastdi, nplusx, nplusy, ier, iter, phase;  // phase 1: knots, 2: p iteration, 0: done
    int ich1, ich3;
    double p, fp, fp0, fpold, reducx, reducy, fpms, p1, f1, p3, f3;
};

// Boundary knots and the ier = -2 flag at the top of each knot-growth iteration (fpregr label 120+).
PMR_HD inline void begin_iteration(Ctl &c, double *tx, double *ty) {
    if (c.nx == c.nminx && c.ny == c.nminy) c.ier = kIerLsqPoly;
    c.nrintx = c.nx - c.nminx + 1;
    c.nrinty = c.ny - c.nminy + 1;
    for (int j = 0; j <= c.kx; j++) {
        tx[j] = 0.0;
        tx[c.nx - 1 - j] = (double)(c.mx - 1);
    }
    for (int j = 0; j <= c.ky; j++) {
        ty[j] = 0.0;
        ty[c.ny - 1 - j] = (double)(c.my - 1);
    }
}

// Input checks of regrid and fpregr's initialisation for iopt = 0, s > 0.  Returns false (ier = 10)
// when the input is refused.
PMR_HD inline bool init(Ctl &c, int mx, int my, int kx, int ky, double s, int nxest, int nyest, int maxit,
                        double *tx, double *ty, const Work &w) {
    c.mx = mx; c.my = my; c.kx = kx; c.ky = ky; c.s = s; c.nxest = nxest; c.nyest = nyest; c.maxit = maxit;
    c.phase = 0;
    c.ier = kIerInput;
    c.nx = c.ny = 0;
    c.fp = 0.0;
    c.nminx = 2 * (kx + 1);
    c.nminy = 2 * (ky + 1);
    if (kx < 1 || kx > kMaxK || ky < 1 || ky > kMaxK || !(s > 0.0) || maxit < 1) return false;
    if (mx < kx + 1 || nxest < c.nminx || my < ky + 1 || nyest < c.nminy) return false;
    c.ier = kIerOk;
    c.acc = kTol * s;
    c.nmaxx = mx + kx + 1;
    c.nmaxy = my + ky + 1;
    c.nxe = c.nmaxx < nxest ? c.nmaxx : nxest;
    c.nye = c.nmaxy < nyest ? c.nmaxy : nyest;
    c.nx = c.nminx;
    c.ny = c.nminy;
    w.nrdatx[0] = mx - 2;
    w.nrdaty[0] = my - 2;
    c.lastdi = 0;
    c.nplusx = c.nplusy = 0;
    c.fp0 = c.fpold = c.reducx = c.reducy = 0.0;
    c.p = -1.0;
    c.iter = 1;
    c.phase = 1;
    begin_iteration(c, tx, ty);
    return true;
}

// fpregr after one fpgrre with fit residual fp: decide the next step.  Returns true when fpgrre must
// run again (new knots in tx / ty, or a new p), false when the fit is final (c.ier, c.fp set).
PMR_HD inline bool after_fit(Ctl &c, double fp, double *tx, double *ty, const Work &w) {
    c.fp = fp;
    if (c.phase == 1) {
        if (c.ier == kIerLsqPoly) c.fp0 = fp;
        c.fpms = fp - c.s;
        bool to_part2 = false;
        if (fabs(c.fpms) < c.acc) {
            c.phase = 0;
            return false;
        }
        if (c.fpms < 0.0) {
            to_part2 = true;
        } else {
            if (c.nx == c.nmaxx && c.ny == c.nmaxy) {
                c.ier = kIerInterp;
                c.fp = 0.0;
                c.phase = 0;
                return false;
            }
            if (c.nx == c.nxe && c.ny == c.nye) {
                c.ier = kIerNest;
                c.phase = 0;
                return false;
            }
            c.ier = kIerOk;
            if (c.lastdi < 0) c.reducx = c.fpold - fp;
            else if (c.lastdi > 0) c.reducy = c.fpold - fp;
            c.fpold = fp;
            int nplx = 1, nply = 1;
            if (c.nx != c.nminx) {
                int npl1 = c.nplusx * 2;
                const double rn = c.nplusx;
                if (c.reducx > c.acc) npl1 = trunc_to_int(div_rn(rn * c.fpms, c.reducx));
                int lo = npl1 > c.nplusx / 2 ? npl1 : c.nplusx / 2;
                if (lo < 1) lo = 1;
                nplx = c.nplusx * 2 < lo ? c.nplusx * 2 : lo;
            }
            if (c.ny != c.nminy) {
                int npl1 = c.nplusy * 2;
                const double rn = c.nplusy;
                if (c.reducy > c.acc) npl1 = trunc_to_int(div_rn(rn * c.fpms, c.reducy));
                int lo = npl1 > c.nplusy / 2 ? npl1 : c.nplusy / 2;
                if (lo < 1) lo = 1;
                nply = c.nplusy * 2 < lo ? c.nplusy * 2 : lo;
            }
            bool addx = nplx < nply || (nplx == nply && c.lastdi >= 0);
            if (addx && c.nx == c.nxe) addx = false;
            else if (!addx && c.ny == c.nye) addx = true;
            if (addx) {
                c.lastdi = -1;
                c.nplusx = nplx;
                for (int l = 0; l < c.nplusx; l++) {
                    fpknot(tx - 1, c.nx, w.fpintx - 1, w.nrdatx - 1, c.nrintx);
                    if (c.nx == c.nxe) break;
                }
                if (c.nx == c.nmaxx) interpolation_knots(tx - 1, c.mx, c.kx);
            } else {
                c.lastdi = 1;
                c.nplusy = nply;
                for (int l = 0; l < c.nplusy; l++) {
                    fpknot(ty - 1, c.ny, w.fpinty - 1, w.nrdaty - 1, c.nrinty);
                    if (c.ny == c.nye) break;
                }
                if (c.ny == c.nmaxy) interpolation_knots(ty - 1, c.my, c.ky);
            }
            c.iter++;
            if (c.iter <= c.mx + c.my) {
                begin_iteration(c, tx, ty);
                return true;
            }
            to_part2 = true;
        }
        if (to_part2) {
            if (c.ier == kIerLsqPoly) {
                c.phase = 0;
                return false;
            }
            c.p1 = 0.0;
            c.f1 = c.fp0 - c.s;
            c.p3 = -1.0;
            c.f3 = c.fpms;
            c.p = 1.0;
            c.ich1 = c.ich3 = 0;
            c.iter = 1;
            c.phase = 2;
            return true;
        }
    }
    // part 2: the root of f(p) = s
    c.fpms = fp - c.s;
    if (fabs(c.fpms) < c.acc) {
        c.phase = 0;
        return false;
    }
    if (c.iter == c.maxit) {
        c.ier = kIerMaxit;
        c.phase = 0;
        return false;
    }
    const double p2 = c.p, f2 = c.fpms;
    c.iter++;
    if (c.ich3 == 0) {
        if (!((f2 - c.f3) > c.acc)) {
            c.p3 = p2;
            c.f3 = f2;
            c.p = c.p * kCon4;
            if (c.p <= c.p1) c.p = c.p1 * kCon9 + p2 * kCon1;
            return true;
        }
        if (f2 < 0.0) c.ich3 = 1;
    }
    if (c.ich1 == 0) {
        if (!((c.f1 - f2) > c.acc)) {
            c.p1 = p2;
            c.f1 = f2;
            c.p = div_rn(c.p, kCon4);
            if (c.p3 < 0.0) return true;
            if (c.p >= c.p3) c.p = p2 * kCon1 + c.p3 * kCon9;
            return true;
        }
        if (f2 > 0.0) c.ich1 = 1;
    }
    if (f2 >= c.f1 || f2 <= c.f3) {
        c.ier = kIerTheory;
        c.phase = 0;
        return false;
    }
    c.p = fprati(c.p1, c.f1, p2, f2, c.p3, c.f3);
    return true;
}

// ---- fpgrre: least-squares (p < 0) or smoothing (p > 0) spline for the current knots ---------------
// Ex runs the parallel pieces: each(n, f) calls f(j) for j < n (any order, any thread), one(f) runs f
// on a single thread, lane(i, f) runs f on thread "i" (independent scalar jobs may run concurrently),
// sync() orders everything before it against everything after it.  Z(i, j) is the data at x = i, y = j.
// rot must hold 3 * (max(kx, ky) + 2) doubles visible to all threads.  Returns nothing; the sums land in
// *fp, w.fpintx and w.fpinty (valid after the final sync).
template <class Ex, class Z>
PMR_HD void fpgrre(const Ex &ex, const Z &z, int mx, int my, int kx, int ky, const double *tx, int nx,
                   const double *ty, int ny, double p, double *c, const Work &w, double *rot, double *fp) {
    const int kx1 = kx + 1, kx2 = kx + 2, ky1 = ky + 1, ky2 = ky + 2;
    const int nk1x = nx - kx1, nk1y = ny - ky1;
    const double pinv = p > 0.0 ? div_rn(1.0, p) : 0.0;
    const double *tx1 = tx - 1, *ty1 = ty - 1;
    // observation matrices (spx), (spy) and, for p > 0, the penalty rows (bx), (by)
    ex.each(mx, [&](int it) {
        const int l = knot_interval(tx1, nx, kx, (double)it);
        fpbspl(tx1, kx, (double)it, l, w.spx + (int64_t)it * kx1);
        w.nrx[it] = l - kx1;
    });
    ex.each(my, [&](int it) {
        const int l = knot_interval(ty1, ny, ky, (double)it);
        fpbspl(ty1, ky, (double)it, l, w.spy + (int64_t)it * ky1);
        w.nry[it] = l - ky1;
    });
    if (p > 0.0 && nx != 2 * kx1) ex.each(nx - 2 * kx1, [&](int r) { fpdisc_row(tx1, nx, kx2, r, w.bx + (int64_t)r * kx2); });
    if (p > 0.0 && ny != 2 * ky1) ex.each(ny - 2 * ky1, [&](int r) { fpdisc_row(ty1, ny, ky2, r, w.by + (int64_t)r * ky2); });
    ex.each(my * nk1x, [&](int i) { w.q[i] = 0.0; });
    ex.each(nk1x * kx2, [&](int i) { w.ax[i] = 0.0; });
    ex.each(nk1x * nk1y, [&](int i) { c[i] = 0.0; });
    ex.each(nk1y * ky2, [&](int i) { w.ay[i] = 0.0; });
    ex.sync();

    // One row (data row of site `it`, or penalty row `nrold`) rotated into the triangle a[][kb2]: the
    // scalar part.  rot[3 i .. 3 i + 2] = (cos, sin, applied) of band element i.
    auto rotate_row = [&](double *a, int kb2, const double *sp, const double *b, int it, int nrold, bool data_row,
                          int iband, int irot) {
        double h[kMaxK + 2];
        if (data_row) {
            h[iband - 1] = 0.0;
            for (int j = 0; j < kb2 - 1; j++) h[j] = sp[(int64_t)it * (kb2 - 1) + j];
        } else {
            for (int j = 0; j < kb2; j++) h[j] = b[(int64_t)nrold * kb2 + j] * pinv;
        }
        for (int i = 0; i < iband; i++) {
            irot++;
            const double piv = h[i];
            rot[3 * i + 2] = 0.0;
            if (piv == 0.0) continue;
            double *arow = a + (int64_t)(irot - 1) * kb2;
            double cs, sn;
            fpgivs(piv, arow[0], cs, sn);
            rot[3 * i] = cs;
            rot[3 * i + 1] = sn;
            rot[3 * i + 2] = 1.0;
            if (i == iband - 1) break;
            for (int j = i + 1, i2 = 1; j < iband; j++, i2++) fprota(cs, sn, h[j], arow[i2]);
        }
    };

    // (ax) -> (rx) with Givens rotations; the same rotations on the my columns of q
    int nrold = 0, ibandx = kx1;
    for (int it = 0; it < mx; it++) {
        const int number = w.nrx[it];
        for (;;) {
            const bool data_row = nrold == number;
            if (!data_row && !(p > 0.0)) {
                nrold++;
                continue;
            }
            if (!data_row) ibandx = kx2;
            const int irot0 = data_row ? number : nrold;
            const int iband = ibandx;
            ex.one([&] { rotate_row(w.ax, kx2, w.spx, w.bx, it, nrold, data_row, iband, irot0); });
            ex.sync();
            ex.each(my, [&](int j) {
                double right = data_row ? z(it, j) : 0.0;
                int irot = irot0;
                for (int i = 0; i < iband; i++) {
                    irot++;
                    if (rot[3 * i + 2] == 0.0) continue;
                    fprota(rot[3 * i], rot[3 * i + 1], right, w.q[(int64_t)(irot - 1) * my + j]);
                }
            });
            ex.sync();
            if (data_row) break;
            nrold++;
        }
    }
    // (ay) -> (ry); the same rotations on the nk1x columns of g (rows of q), into c
    nrold = 0;
    int ibandy = ky1;
    for (int it = 0; it < my; it++) {
        const int number = w.nry[it];
        for (;;) {
            const bool data_row = nrold == number;
            if (!data_row && !(p > 0.0)) {
                nrold++;
                continue;
            }
            if (!data_row) ibandy = ky2;
            const int irot0 = data_row ? number : nrold;
            const int iband = ibandy;
            ex.one([&] { rotate_row(w.ay, ky2, w.spy, w.by, it, nrold, data_row, iband, irot0); });
            ex.sync();
            ex.each(nk1x, [&](int j) {
                double right = data_row ? w.q[(int64_t)j * my + it] : 0.0;
                int irot = irot0;
                for (int i = 0; i < iband; i++) {
                    irot++;
                    if (rot[3 * i + 2] == 0.0) continue;
                    fprota(rot[3 * i], rot[3 * i + 1], right, c[(int64_t)j * nk1y + irot - 1]);
                }
            });
            ex.sync();
            if (data_row) break;
            nrold++;
        }
    }
    // (ry) c (rx)' = h: back substitution along y (per x row), then along x (per y column)
    ex.each(nk1x, [&](int i) { fpback_inplace(w.ay, ky2, c + (int64_t)i * nk1y, 1, nk1y, ibandy); });
    ex.sync();
    ex.each(nk1y, [&](int j) { fpback_inplace(w.ax, kx2, c + j, nk1y, nk1x, ibandx); });
    ex.sync();
    // squared residuals, then fp, fpx, fpy each summed in fpgrre's order
    ex.each(mx * my, [&](int idx) {
        const int i1 = idx / my, i2 = idx - i1 * my;
        double term = 0.0;
        int k1 = w.nrx[i1] * nk1y + w.nry[i2];
        for (int l1 = 0; l1 < kx1; l1++) {
            int k2 = k1;
            const double fac = w.spx[(int64_t)i1 * kx1 + l1];
            for (int l2 = 0; l2 < ky1; l2++) {
                term = term + fac * w.spy[(int64_t)i2 * ky1 + l2] * c[k2];
                k2++;
            }
            k1 += nk1y;
        }
        const double r = z(i1, i2) - term;
        w.term[idx] = r * r;
    });
    ex.sync();
    ex.lane(0, [&] {
        double s = 0.0;
        for (int64_t i = 0; i < (int64_t)mx * my; i++) s = s + w.term[i];
        *fp = s;
    });
    ex.lane(1, [&] {
        double *fpx = w.fpintx;
        for (int i = 0; i < nx; i++) fpx[i] = 0.0;
        int nroldx = 0;
        for (int i1 = 0; i1 < mx; i1++) {
            const int numx = w.nrx[i1];
            for (int i2 = 0; i2 < my; i2++) {
                const double term = w.term[(int64_t)i1 * my + i2];
                fpx[numx] = fpx[numx] + term;
                if (numx != nroldx) {
                    const double fac = term * 0.5;
                    fpx[numx] = fpx[numx] - fac;
                    fpx[numx - 1] = fpx[numx - 1] + fac;
                }
            }
            nroldx = numx;
        }
    });
    ex.lane(2, [&] {
        double *fpy = w.fpinty;
        for (int i = 0; i < ny; i++) fpy[i] = 0.0;
        for (int i1 = 0; i1 < mx; i1++) {
            int nroldy = 0;
            for (int i2 = 0; i2 < my; i2++) {
                const double term = w.term[(int64_t)i1 * my + i2];
                const int numy = w.nry[i2];
                fpy[numy] = fpy[numy] + term;
                if (numy != nroldy) {
                    const double fac = term * 0.5;
                    fpy[numy] = fpy[numy] - fac;
                    fpy[numy - 1] = fpy[numy - 1] + fac;
                }
                nroldy = numy;
            }
        }
    });
    ex.sync();
}

// ---- the whole fit of one plane --------------------------------------------------------------------
// Outputs: tx[nxest], ty[nyest], c[(nxest-kx-1)(nyest-ky-1)], out_n = {nx, ny, ier}, *out_fp.
// ctl, rot and fp_slot must be visible to all threads of Ex (shared memory on the device).
template <class Ex, class Z>
PMR_HD void fit_plane(const Ex &ex, const Z &z, int mx, int my, int kx, int ky, double s, int nxest, int nyest,
                      int maxit, double *tx, double *ty, double *c, const Work &w, Ctl &ctl, double *rot,
                      double *fp_slot, int *out_n, double *out_fp) {
    ex.one([&] { init(ctl, mx, my, kx, ky, s, nxest, nyest, maxit, tx, ty, w); });
    ex.sync();
    bool more = ctl.phase != 0;
    while (more) {
        fpgrre(ex, z, mx, my, kx, ky, tx, ctl.nx, ty, ctl.ny, ctl.p, c, w, rot, fp_slot);
        ex.one([&] { after_fit(ctl, *fp_slot, tx, ty, w); });
        ex.sync();
        more = ctl.phase != 0;
    }
    ex.one([&] {
        out_n[0] = ctl.nx;
        out_n[1] = ctl.ny;
        out_n[2] = ctl.ier;
        *out_fp = ctl.fp;
    });
}

// ---- evaluation: fpbisp for one point (bispeu), knots / coefficients of one plane -------------------
PMR_HD inline double evaluate(const double *tx, int nx, const double *ty, int ny, const double *c, int kx, int ky,
                              double x, double y) {
    const double *tx1 = tx - 1, *ty1 = ty - 1;
    const int kx1 = kx + 1, ky1 = ky + 1, nky1 = ny - ky1;
    double arg = x;
    if (arg < tx1[kx1]) arg = tx1[kx1];
    if (arg > tx1[nx - kx]) arg = tx1[nx - kx];
    const int lx = knot_interval(tx1, nx, kx, arg);
    double wx[kMaxK + 1], wy[kMaxK + 1];
    fpbspl(tx1, kx, arg, lx, wx);
    arg = y;
    if (arg < ty1[ky1]) arg = ty1[ky1];
    if (arg > ty1[ny - ky]) arg = ty1[ny - ky];
    const int ly = knot_interval(ty1, ny, ky, arg);
    fpbspl(ty1, ky, arg, ly, wy);
    int l1 = (lx - kx1) * nky1 + (ly - ky1);
    double sp = 0.0;
    for (int i1 = 0; i1 < kx1; i1++) {
        int l2 = l1;
        for (int j1 = 0; j1 < ky1; j1++) {
            sp = sp + c[l2] * wx[i1] * wy[j1];
            l2++;
        }
        l1 += nky1;
    }
    return sp;
}

}  // namespace regrid
}  // namespace pm
