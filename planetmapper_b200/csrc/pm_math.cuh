// pm_math.cuh - FP64 primitives tuned for the sm_100a FP64 pipe.
//
// Why not CUDA's libm here: the first version of the backplane kernel (profiles/
// r1_summary.md) spent two thirds of its issue slots outside the FP64 pipe - 64-bit
// polynomial coefficients materialised as UMOV/IMAD pairs, slow-path CALLs for div /
// sqrt / trig range reduction, 161 KB of straight-line code missing the instruction
// cache.  The routines below
//   * seed division and square root with one MUFU (rcp.approx / rsqrt.approx.f64,
//     ~20 good bits) and finish with a cubically convergent FMA step (no slow path:
//     every operand on the hot path is a finite, normal, kilometre-scale number),
//   * keep polynomial coefficients in __constant__ tables so a DFMA reads them as
//     c[bank][offset] operands instead of moving immediates into registers,
//   * use argument ranges the geometry guarantees (|angle| <= pi/4 for pixel offsets
//     and frame spins) and leave everything else to a cold, non-inlined fallback.
// Accuracy is <= 1-2 ulp for every routine (tests/test_device_math.py measures it on
// the host build, tests/test_gpu_math.py on the GPU), i.e. five orders of magnitude
// inside the 1e-9 deg parity bar.
//
// The header also compiles for the host (nvcc host pass) so that tests can run the
// very same per-pixel code against the oracle without a GPU; the MUFU seeds are then
// emulated by truncating an exact result to 20 mantissa bits.  The product never
// executes the host instantiation (no CPU fallback): libpm_b200.so only exports
// launchers of __global__ kernels.
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define PM_HD __host__ __device__ __forceinline__
#define PM_HD_NOINLINE static __host__ __device__ __noinline__
#define PM_DEV_TABLE(name, n, ...)                        \
    static __constant__ __align__(16) double name##_dev[n] = {__VA_ARGS__}; \
    static const double name##_host[n] = {__VA_ARGS__};
#else
#define PM_HD inline
#define PM_HD_NOINLINE static
#define PM_DEV_TABLE(name, n, ...) static const double name##_host[n] = {__VA_ARGS__};
#endif

#ifdef __CUDA_ARCH__
#define PM_T(name) name##_dev
#else
#define PM_T(name) name##_host
#endif

namespace pm {

constexpr double kPi = 3.14159265358979323846264338327950288;
constexpr double kTwoPi = 2.0 * kPi;
constexpr double kHalfPi = 0.5 * kPi;
constexpr double kQuarterPi = 0.25 * kPi;
constexpr double kDpr = 180.0 / kPi;
constexpr double kRpd = kPi / 180.0;

// minimax fits (mpmath, Chebyshev nodes, 60 digits; tools/fit_coefficients.py):
//   atan(q) = q + q z A(z),  z = q^2 <= tan(pi/12)^2     |err| < 2e-17
//   sin(x)  = x + x z S(z),  z = x^2 <= (pi/4)^2          |err| < 2e-17
//   cos(x)  = 1 - z/2 + z^2 C(z)                           |err| < 5e-19
PM_DEV_TABLE(kAtanC, 8, -0.33333333333333245175, 0.19999999999842781854, -0.14285714239619743943,
             0.11111105950225735071, -0.090906243717563017737, 0.076837307398386464706,
             -0.065219990167523964706, 0.04578335659104139954)
PM_DEV_TABLE(kSinC, 6, -0.16666666666666664621, 0.008333333333330946103, -0.00019841269836754970194,
             2.7557316100683122624e-6, -2.5051131455447427132e-8, 1.5918101231677278624e-10)
PM_DEV_TABLE(kCosC, 6, 0.041666666666666665387, -0.0013888888888887395746, 0.000024801587298763433277,
             -2.7557317270560382548e-7, 2.0876146024701932874e-9, -1.1382614869434128293e-11)
// misc constants read as constant-bank operands: tan(pi/12), pi/4, pi/2, pi, 2/pi,
// pi/2 split (hi, lo), 2 pi, 1/(2 pi), sqrt(3), pi/6, the zero guard of the square roots
PM_DEV_TABLE(kMisc, 12, 0.2679491924311227064725537, 0.78539816339744830961566, 1.5707963267948966192313,
             3.1415926535897932384626, 0.6366197723675813430755351, 1.570796326794896619231322,
             6.12323399573676588613033e-17, 6.283185307179586476925287, 0.1591549430918953357688838,
             1.732050807568877293527446, 0.5235987755982988730771072, 1.0e-300)

// x + sqrt_guard() keeps an rsqrt seed finite at x == 0 (1e-300, read from the table like the other
// full-mantissa literals instead of being rebuilt by two 32-bit moves at every use)
PM_HD double sqrt_guard() { return PM_T(kMisc)[11]; }

// ---- MUFU seeds ----------------------------------------------------------------
PM_HD double rcp_seed(double b) {
#ifdef __CUDA_ARCH__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    return r;
#else
    uint64_t u;
    memcpy(&u, &b, 8);
    u &= 0xFFFFFFFF00000000ull;
    double bt;
    memcpy(&bt, &u, 8);
    double r = 1.0 / bt;
    memcpy(&u, &r, 8);
    u &= 0xFFFFFFFF00000000ull;
    memcpy(&r, &u, 8);
    return r;
#endif
}
PM_HD double rsqrt_seed(double x) {
#ifdef __CUDA_ARCH__
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return r;
#else
    uint64_t u;
    memcpy(&u, &x, 8);
    u &= 0xFFFFFFFF00000000ull;
    double xt;
    memcpy(&xt, &u, 8);
    double r = 1.0 / ::sqrt(xt);
    memcpy(&u, &r, 8);
    u &= 0xFFFFFFFF00000000ull;
    memcpy(&r, &u, 8);
    return r;
#endif
}

// 1 / b for finite normal b != 0 (no denormal / inf / zero slow path)
PM_HD double fast_rcp(double b) {
    double r = rcp_seed(b);
    double e = fma(-b, r, 1.0);  // |e| <~ 2^-19
    e = fma(e, e, e);            // e + e^2: cubic convergence, residual e^3 ~ 2^-57
    return fma(r, e, r);
}
// a / b, correctly rounded in all but a vanishing fraction of cases
PM_HD double fast_div(double a, double b) {
    double r = fast_rcp(b);
    double q = a * r;
    double rem = fma(-b, q, a);
    return fma(rem, r, q);
}
// 1 / sqrt(x) for finite normal x > 0
PM_HD double fast_rsqrt(double x) {
    double y = rsqrt_seed(x);
    double xy = x * y;
    double e = fma(-xy, y, 1.0);       // 1 - x y^2
    double p = fma(0.375, e, 0.5);     // y (1 + e/2 + 3 e^2 / 8): residual 5/16 e^3
    return fma(y, p * e, y);
}
// sqrt(x) for x >= 0 (x == 0 -> 0).  Not for negative x (see fast_sqrt_nan).
PM_HD double fast_sqrt(double x) {
    double y = fast_rsqrt(x + sqrt_guard());
    double s = x * y;
    double rem = fma(-s, s, x);
    return fma(rem, 0.5 * y, s);
}
// Two-instruction-cheaper variants (<= 1.5 ulp instead of <= 0.5) for values that feed light
// times, angle arguments and normalisations, where the last half ulp is immaterial
PM_HD double fast_sqrt_lite(double x) { return x * fast_rsqrt(x + sqrt_guard()); }
// ... for x known to be finite, normal and > 0 (lengths of vectors that cannot vanish): no zero guard
PM_HD double fast_sqrt_pos(double x) { return x * fast_rsqrt(x); }
PM_HD double fast_div_lite(double a, double b) { return a * fast_rcp(b); }
// sqrt that keeps IEEE's NaN for negative input
PM_HD double fast_sqrt_nan(double x) { return (x < 0.0) ? NAN : fast_sqrt_lite(x); }

// ---- trig ----------------------------------------------------------------------
// sin, cos for |x| <= pi/4 (no range reduction)
PM_HD void sincos_quarter(double x, double &s, double &c) {
    const double z = x * x;
    double ps = PM_T(kSinC)[5];
    double pc = PM_T(kCosC)[5];
#pragma unroll
    for (int i = 4; i >= 0; i--) {
        ps = fma(ps, z, PM_T(kSinC)[i]);
        pc = fma(pc, z, PM_T(kCosC)[i]);
    }
    s = fma(x * z, ps, x);
    c = fma(z * z, pc, fma(-0.5, z, 1.0));
}
// library fallback, kept out of line so the hot code stays small
PM_HD_NOINLINE void sincos_lib(double x, double *s, double *c) {
#ifdef __CUDA_ARCH__
    ::sincos(x, s, c);
#else
    *s = ::sin(x);
    *c = ::cos(x);
#endif
}
// sin, cos for small arguments with a cold fallback for everything else
PM_HD void sincos_small(double x, double &s, double &c) {
    if (fabs(x) <= PM_T(kMisc)[1]) {
        sincos_quarter(x, s, c);
    } else {
        sincos_lib(x, &s, &c);
    }
}
// sin, cos for |x| <= 2^-8: x + x z (-1/6 + z/120), 1 - z/2 + z^2 (1/24 - z/720); the first omitted terms
// are < 1e-18 relative.  Pixel offsets from the optical axis of a telescope image (an arcminute field is
// 3e-4 rad) stay far inside this range.
// [0] 1/120, [1] -1/720, [2] -1/6, [3] 1/24 (also the spin series of pm_device.cuh's make_rot)
PM_DEV_TABLE(kTinyC, 4, 1.0 / 120.0, -1.0 / 720.0, -1.0 / 6.0, 1.0 / 24.0)
PM_HD void sincos_tiny(double x, double &s, double &c) {
    const double z = x * x;
    s = fma(x * z, fma(z, PM_T(kTinyC)[0], PM_T(kTinyC)[2]), x);
    c = fma(z * z, fma(z, PM_T(kTinyC)[1], PM_T(kTinyC)[3]), fma(-0.5, z, 1.0));
}
// sin, cos of two small angles with ONE range test, so that the four polynomial
// chains share a basic block (cold library fallback for anything above pi/4)
PM_HD void sincos_small2(double a, double b, double &sa, double &ca, double &sb, double &cb) {
    const double m = fmax(fabs(a), fabs(b));
    if (m <= 0.00390625) {  // 2^-8
        sincos_tiny(a, sa, ca);
        sincos_tiny(b, sb, cb);
    } else if (m <= PM_T(kMisc)[1]) {
        sincos_quarter(a, sa, ca);
        sincos_quarter(b, sb, cb);
    } else {
        sincos_lib(a, &sa, &ca);
        sincos_lib(b, &sb, &cb);
    }
}
// sin, cos for |x| < ~1e5 (two-term Cody-Waite with FMA), cold fallback beyond
PM_HD void sincos_full(double x, double &s, double &c) {
    if (!(fabs(x) < 1.0e5)) {
        sincos_lib(x, &s, &c);
        return;
    }
    const double k = rint(x * PM_T(kMisc)[4]);
    double r = fma(-k, PM_T(kMisc)[5], x);
    r = fma(-k, PM_T(kMisc)[6], r);
    double sr, cr;
    sincos_quarter(r, sr, cr);
    const int n = (int)k;
    if (n & 1) {
        double t = sr;
        sr = cr;
        cr = -t;
    }
    if (n & 2) {
        sr = -sr;
        cr = -cr;
    }
    s = sr;
    c = cr;
}

// Bit-level helpers: keep sign / magnitude bookkeeping off the FP64 pipe
PM_HD bool pos_gt(double a, double b) {  // a > b for non-NaN a, b >= 0 (IEEE ordering == integer ordering)
#ifdef __CUDA_ARCH__
    return __double_as_longlong(a) > __double_as_longlong(b);
#else
    return a > b;
#endif
}
PM_HD double with_sign_of(double r, double y) {  // r >= 0: copysign(r, y)
#ifdef __CUDA_ARCH__
    const int hi = __double2hiint(r) | (__double2hiint(y) & 0x80000000);
    return __hiloint2double(hi, __double2loint(r));
#else
    return copysign(r, y);
#endif
}
PM_HD double abs_bits(double x) {  // fabs(x) as one integer AND of the high word instead of an FP64 DADD
#ifdef __CUDA_ARCH__
    return __hiloint2double(__double2hiint(x) & 0x7fffffff, __double2loint(x));
#else
    return fabs(x);
#endif
}
PM_HD bool sign_bit(double x) {
#ifdef __CUDA_ARCH__
    return __double2hiint(x) < 0;
#else
    return signbit(x);
#endif
}

// atan(a / b) for 0 <= a <= b, b > 0: one division; the argument is folded into
// |q| <= tan(pi/12) by  atan(a/b) = pi/6 + atan((sqrt(3) a - b) / (sqrt(3) b + a)).
// Branch-free on purpose: independent calls then sit in one basic block and the
// scheduler interleaves their dependent FMA chains.
PM_HD double atan_ratio(double mn, double mx) {
    const bool hi = mn > mx * PM_T(kMisc)[0];
    const double num = hi ? fma(PM_T(kMisc)[9], mn, -mx) : mn;
    const double den = hi ? fma(PM_T(kMisc)[9], mx, mn) : mx;
    const double q = fast_div_lite(num, den);
    const double z = q * q;
    double p = PM_T(kAtanC)[7];
#pragma unroll
    for (int i = 6; i >= 0; i--) p = fma(p, z, PM_T(kAtanC)[i]);
    double r = fma(q * z, p, q);
    if (hi) r += PM_T(kMisc)[10];
    return r;
}
// atan2(y, x), full quadrant, atan2(0, 0) = 0 (the convention recrad / reclat / recgeo
// apply explicitly).  NaN in -> NaN out.
PM_HD double fast_atan2(double y, double x) {
    const double ax = abs_bits(x), ay = abs_bits(y);
    const bool sw = pos_gt(ay, ax);
    const double mx = sw ? ay : ax, mn = sw ? ax : ay;
    double r = atan_ratio(mn, mx);  // 0 / 0 -> NaN, replaced below
    if (sw) r = PM_T(kMisc)[2] - r;
    if (sign_bit(x)) r = PM_T(kMisc)[3] - r;
    r = with_sign_of(r, y);
    return (mx == 0.0) ? 0.0 : r;
}
// atan2(y, x) for y >= 0 and (x, y) != (0, 0): angle in [0, pi] (vector separations)
PM_HD double fast_atan2_ypos(double y, double x) {
    const double ax = abs_bits(x);
    const bool sw = pos_gt(abs_bits(y), ax);
    const double mx = sw ? y : ax, mn = sw ? ax : y;
    double r = atan_ratio(mn, mx);
    if (sw) r = PM_T(kMisc)[2] - r;
    if (sign_bit(x)) r = PM_T(kMisc)[3] - r;
    return r;
}
// atan2(y, x) for x >= 0 and (x, y) != (0, 0): angle in [-pi/2, pi/2] (latitudes)
PM_HD double fast_atan2_xpos(double y, double x) {
    const double ay = abs_bits(y);
    const bool sw = pos_gt(ay, abs_bits(x));
    const double mx = sw ? ay : x, mn = sw ? x : ay;
    double r = atan_ratio(mn, mx);
    if (sw) r = PM_T(kMisc)[2] - r;
    return with_sign_of(r, y);
}
// acos(x); NaN for |x| > 1 like the libm routine
PM_HD double fast_acos(double x) {
    return fast_atan2_ypos(fast_sqrt_nan((1.0 - x) * (1.0 + x)), x);
}

}  // namespace pm
