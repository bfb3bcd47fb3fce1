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
// tables indexed per lane: global memory read through the read-only cache (a __constant__ operand
// serialises a warp over its distinct addresses)
#define PM_LDG_TABLE(name, n, ...)                        \
    static __device__ __align__(16) double name##_dev[n] = {__VA_ARGS__}; \
    static const double name##_host[n] = {__VA_ARGS__};
#else
#define PM_HD inline
#define PM_HD_NOINLINE static
#define PM_DEV_TABLE(name, n, ...) static const double name##_host[n] = {__VA_ARGS__};
#define PM_LDG_TABLE(name, n, ...) static const double name##_host[n] = {__VA_ARGS__};
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
//   sin(x)  = x + x z S(z),  z = x^2 <= (pi/4)^2          |err| < 2e-17
//   cos(x)  = 1 - z/2 + z^2 C(z)                           |err| < 5e-19
PM_DEV_TABLE(kSinC, 6, -0.16666666666666664621, 0.008333333333330946103, -0.00019841269836754970194,
             2.7557316100683122624e-6, -2.5051131455447427132e-8, 1.5918101231677278624e-10)
PM_DEV_TABLE(kCosC, 6, 0.041666666666666665387, -0.0013888888888887395746, 0.000024801587298763433277,
             -2.7557317270560382548e-7, 2.0876146024701932874e-9, -1.1382614869434128293e-11)
// misc constants read as constant-bank operands: pi/4, pi/2, pi, 2/pi, pi/2 split (hi, lo), 2 pi,
// 1/(2 pi), the zero guard of the square roots
PM_DEV_TABLE(kMisc, 9, 0.78539816339744830961566, 1.5707963267948966192313, 3.1415926535897932384626,
             0.6366197723675813430755351, 1.570796326794896619231322, 6.12323399573676588613033e-17,
             6.283185307179586476925287, 0.1591549430918953357688838, 1.0e-300)

// x + sqrt_guard() keeps an rsqrt seed finite at x == 0 (1e-300, read from the table like the other
// full-mantissa literals instead of being rebuilt by two 32-bit moves at every use)
PM_HD double sqrt_guard() { return PM_T(kMisc)[8]; }

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
    if (fabs(x) <= PM_T(kMisc)[0]) {
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
    } else if (m <= PM_T(kMisc)[0]) {
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
    const double k = rint(x * PM_T(kMisc)[3]);
    double r = fma(-k, PM_T(kMisc)[4], x);
    r = fma(-k, PM_T(kMisc)[5], r);
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

// Table-reduced arctangent (tools/fit_atan_table.py): series, and (t0, atan(t0)) at t0 = k / 256
// atan(r) = r + r z (c1 + c2 z + c3 z^2), |r| <= 2^-8: relative truncation error 6.02e-21
PM_DEV_TABLE(kAtanC, 3, -0.3333333333333333, 0.2, -0.14285714285714285)
// (k / 2^8, atan(k / 2^8)) for k = 0 .. 256
PM_LDG_TABLE(kAtanT, 514,
             0.0, 0.0,
             0.00390625, 0.0039062301319669718,
             0.0078125, 0.007812341060101111,
             0.01171875, 0.01171821360239413,
             0.015625, 0.015623728620476831,
             0.01953125, 0.019528767041413708,
             0.0234375, 0.023433209879467586,
             0.02734375, 0.027336938257824413,
             0.03125, 0.031239833430268277,
             0.03515625, 0.03514177680279678,
             0.0390625, 0.03904264995516699,
             0.04296875, 0.04294233466236217,
             0.046875, 0.046840712915969654,
             0.05078125, 0.05073766694546022,
             0.0546875, 0.05463307923935948,
             0.05859375, 0.05852683256630177,
             0.0625, 0.06241880999595735,
             0.06640625, 0.06630889491982349,
             0.0703125, 0.07019697107187052,
             0.07421875, 0.07408292254903373,
             0.078125, 0.0779666338315423,
             0.08203125, 0.08184798980307655,
             0.0859375, 0.08572687577074481,
             0.08984375, 0.08960317748487175,
             0.09375, 0.09347678115858947,
             0.09765625, 0.09734757348722367,
             0.1015625, 0.10121544166746667,
             0.10546875, 0.10508027341632953,
             0.109375, 0.10894195698986579,
             0.11328125, 0.11280038120165939,
             0.1171875, 0.11665543544106935,
             0.12109375, 0.12050700969122456,
             0.125, 0.12435499454676144,
             0.12890625, 0.12819928123129815,
             0.1328125, 0.13203976161463876,
             0.13671875, 0.1358763282297013,
             0.140625, 0.13970887428916365,
             0.14453125, 0.14353729370182122,
             0.1484375, 0.14736148108865163,
             0.15234375, 0.15118133179858007,
             0.15625, 0.15499674192394097,
             0.16015625, 0.15880760831563107,
             0.1640625, 0.16261382859794857,
             0.16796875, 0.16641530118311493,
             0.171875, 0.1702119252854744,
             0.17578125, 0.1740036009353677,
             0.1796875, 0.17779022899267607,
             0.18359375, 0.18157171116003218,
             0.1875, 0.18534794999569476,
             0.19140625, 0.189118848926084,
             0.1953125, 0.19288431225797467,
             0.19921875, 0.196644245190345,
             0.203125, 0.2003985538258785,
             0.20703125, 0.20414714518211702,
             0.2109375, 0.207889927202263,
             0.21484375, 0.21162680876562978,
             0.21875, 0.21535769969773805,
             0.22265625, 0.21908251078005778,
             0.2265625, 0.22280115375939452,
             0.23046875, 0.22651354135691962,
             0.234375, 0.23021958727684372,
             0.23828125, 0.23391920621473344,
             0.2421875, 0.23761231386547124,
             0.24609375, 0.24129882693085883,
             0.25, 0.24497866312686414,
             0.25390625, 0.24865174119051325,
             0.2578125, 0.2523179808864272,
             0.26171875, 0.25597730301300553,
             0.265625, 0.2596296294082575,
             0.26953125, 0.2632748829552824,
             0.2734375, 0.26691298758740045,
             0.27734375, 0.2705438682929366,
             0.28125, 0.2741674511196588,
             0.28515625, 0.27778366317887326,
             0.2890625, 0.28139243264917846,
             0.29296875, 0.2849936887798813,
             0.296875, 0.2885873618940774,
             0.30078125, 0.29217338339139876,
             0.3046875, 0.29575168575043154,
             0.30859375, 0.29932220253080744,
             0.3125, 0.3028848683749714,
             0.31640625, 0.3064396190096301,
             0.3203125, 0.30998639124688343,
             0.32421875, 0.3135251229850439,
             0.328125, 0.31705575320914703,
             0.33203125, 0.320578221991157,
             0.3359375, 0.3240924704898717,
             0.33984375, 0.32759844095053087,
             0.34375, 0.3310960767041321,
             0.34765625, 0.334585322166459,
             0.3515625, 0.33806612283682547,
             0.35546875, 0.3415384252965417,
             0.359375, 0.34500217720710513,
             0.36328125, 0.34845732730812207,
             0.3671875, 0.3519038254149648,
             0.37109375, 0.35534162241616835,
             0.375, 0.35877067027057225,
             0.37890625, 0.3621909220042122,
             0.3828125, 0.3656023317069669,
             0.38671875, 0.3690048545289644,
             0.390625, 0.3723984466767542,
             0.39453125, 0.37578306540924894,
             0.3984375, 0.3791586690334418,
             0.40234375, 0.38252521689990515,
             0.40625, 0.38588266939807375,
             0.41015625, 0.3892309879513207,
             0.4140625, 0.3925701350118286,
             0.41796875, 0.3959000740552629,
             0.421875, 0.39922076957525254,
             0.42578125, 0.4025321870776825,
             0.4296875, 0.4058342930748041,
             0.43359375, 0.4091270550791683,
             0.4375, 0.4124104415973873,
             0.44140625, 0.4156844221237294,
             0.4453125, 0.41894896713355284,
             0.44921875, 0.4222040480765836,
             0.453125, 0.42544963737004227,
             0.45703125, 0.4286857083916258,
             0.4609375, 0.4319122354723482,
             0.46484375, 0.43512919388924687,
             0.46875, 0.43833655985795783,
             0.47265625, 0.44153431052516673,
             0.4765625, 0.44472242396093936,
             0.48046875, 0.4479008791509373,
             0.484375, 0.4510696559885235,
             0.48828125, 0.4542287352667625,
             0.4921875, 0.4573780986703208,
             0.49609375, 0.4605177287672711,
             0.5, 0.4636476090008061,
             0.50390625, 0.4667677236808665,
             0.5078125, 0.46987805797568694,
             0.51171875, 0.4729785979032656,
             0.515625, 0.4760693303227612,
             0.51953125, 0.47915024292582253,
             0.5234375, 0.48222132422785374,
             0.52734375, 0.4852825635592213,
             0.53125, 0.48833395105640554,
             0.53515625, 0.4913754776531019,
             0.5390625, 0.49440713507127537,
             0.54296875, 0.49742891581217225,
             0.546875, 0.5004408131472942,
             0.55078125, 0.5034428211093364,
             0.5546875, 0.5064349344830967,
             0.55859375, 0.5094171487963564,
             0.5625, 0.5123894603107377,
             0.56640625, 0.5153518660125433,
             0.5703125, 0.518304363603578,
             0.57421875, 0.5212469514919582,
             0.578125, 0.5241796287829132,
             0.58203125, 0.5271023952695796,
             0.5859375, 0.5300152514237931,
             0.58984375, 0.5329181983868821,
             0.59375, 0.5358112379604637,
             0.59765625, 0.5386943725972466,
             0.6015625, 0.541567605391845,
             0.60546875, 0.5444309400716031,
             0.609375, 0.5472843809874369,
             0.61328125, 0.5501279331046931,
             0.6171875, 0.5529616019940283,
             0.62109375, 0.5557853938223135,
             0.625, 0.5585993153435624,
             0.62890625, 0.5614033738898894,
             0.6328125, 0.5641975773624976,
             0.63671875, 0.5669819342227005,
             0.640625, 0.5697564534829784,
             0.64453125, 0.5725211446980724,
             0.6484375, 0.5752760179561178,
             0.65234375, 0.5780210838698195,
             0.65625, 0.5807563535676704,
             0.66015625, 0.5834818386852149,
             0.6640625, 0.5861975513563606,
             0.66796875, 0.5889035042047381,
             0.671875, 0.5915997103351114,
             0.67578125, 0.5942861833248413,
             0.6796875, 0.5969629372154015,
             0.68359375, 0.5996299865039514,
             0.6875, 0.6022873461349642,
             0.69140625, 0.604935031491914,
             0.6953125, 0.6075730583890224,
             0.69921875, 0.6102014430630652,
             0.703125, 0.6128202021652414,
             0.70703125, 0.6154293527531051,
             0.7109375, 0.6180289122825618,
             0.71484375, 0.6206188985999295,
             0.71875, 0.6231993299340659,
             0.72265625, 0.6257702248885632,
             0.7265625, 0.6283316024340097,
             0.73046875, 0.630883481900322,
             0.734375, 0.6334258829691446,
             0.73828125, 0.6359588256663214,
             0.7421875, 0.6384823303544376,
             0.74609375, 0.6409964177254321,
             0.75, 0.6435011087932844,
             0.75390625, 0.6459964248867716,
             0.7578125, 0.6484823876423006,
             0.76171875, 0.6509590189968124,
             0.765625, 0.6534263411807619,
             0.76953125, 0.6558843767111708,
             0.7734375, 0.658333148384756,
             0.77734375, 0.6607726792711327,
             0.78125, 0.6632029927060933,
             0.78515625, 0.665624112284961,
             0.7890625, 0.6680360618560202,
             0.79296875, 0.6704388655140214,
             0.796875, 0.6728325475937632,
             0.80078125, 0.6752171326637499,
             0.8046875, 0.6775926455199252,
             0.80859375, 0.6799591111794819,
             0.8125, 0.6823165548747481,
             0.81640625, 0.684665002047149,
             0.8203125, 0.687004478341245,
             0.82421875, 0.6893350095988459,
             0.828125, 0.6916566218531999,
             0.83203125, 0.6939693413232598,
             0.8359375, 0.6962731944080236,
             0.83984375, 0.69856820768095,
             0.84375, 0.7008544078844502,
             0.84765625, 0.7031318219244538,
             0.8515625, 0.705400476865049,
             0.85546875, 0.7076603999231981,
             0.859375, 0.7099116184635249,
             0.86328125, 0.7121541599931787,
             0.8671875, 0.714388052156769,
             0.87109375, 0.7166133227313746,
             0.875, 0.7188299996216245,
             0.87890625, 0.7210381108548516,
             0.8828125, 0.7232376845763179,
             0.88671875, 0.7254287490445107,
             0.890625, 0.7276113326265107,
             0.89453125, 0.7297854637934291,
             0.8984375, 0.7319511711159166,
             0.90234375, 0.7341084832597397,
             0.90625, 0.7362574289814281,
             0.91015625, 0.7383980371239895,
             0.9140625, 0.7405303366126927,
             0.91796875, 0.7426543564509179,
             0.921875, 0.7447701257160751,
             0.92578125, 0.7468776735555875,
             0.9296875, 0.7489770291829414,
             0.93359375, 0.7510682218738024,
             0.9375, 0.7531512809621944,
             0.94140625, 0.7552262358367449,
             0.9453125, 0.7572931159369924,
             0.94921875, 0.759351950749758,
             0.953125, 0.7614027698055784,
             0.95703125, 0.7634456026752018,
             0.9609375, 0.7654804789661445,
             0.96484375, 0.7675074283193083,
             0.96875, 0.7695264804056583,
             0.97265625, 0.7715376649229596,
             0.9765625, 0.7735410115925735,
             0.98046875, 0.7755365501563117,
             0.984375, 0.7775243103733478,
             0.98828125, 0.7795043220171863,
             0.9921875, 0.7814766148726883,
             0.99609375, 0.7834412187331518,
             1.0, 0.7853981633974483)

PM_HD uint32_t lo_word(double x) {
#ifdef __CUDA_ARCH__
    return (uint32_t)__double2loint(x);
#else
    uint64_t u;
    memcpy(&u, &x, 8);
    return (uint32_t)u;
#endif
}
// atan(a / b) for 0 <= a <= b, b > 0: atan(t0) + atan(r), r = (a - t0 b) / (b + t0 a), one division.
// k = round(256 a / b) from the reciprocal seed: adding 1.5 * 2^44 (ulp 2^-8) leaves it in the low
// mantissa word.  A seed ~20 bits short can move k by one, which keeps |r| <= 2^-8, the range of the
// series.  The clamp keeps a NaN quotient (0 / 0, NaN in) inside the table; the result is NaN anyway.
// Branch-free on purpose: independent calls then sit in one basic block and the scheduler interleaves
// their dependent FMA chains.
PM_HD double atan_ratio(double mn, double mx) {
    const uint32_t kr = lo_word(fma(mn, rcp_seed(mx), 26388279066624.0));
    const uint32_t k = kr < 256u ? kr : 256u;
#ifdef __CUDA_ARCH__
    const double2 e = __ldg(reinterpret_cast<const double2 *>(kAtanT_dev) + k);
    const double t0 = e.x, a0 = e.y;
#else
    const double t0 = kAtanT_host[2 * k], a0 = kAtanT_host[2 * k + 1];
#endif
    const double r = fast_div_lite(fma(-t0, mx, mn), fma(t0, mn, mx));
    const double z = r * r;
    const double p = fma(fma(PM_T(kAtanC)[2], z, PM_T(kAtanC)[1]), z, PM_T(kAtanC)[0]);
    return a0 + fma(r * z, p, r);
}
// atan2(y, x), full quadrant, atan2(0, 0) = 0 (the convention recrad / reclat / recgeo
// apply explicitly).  NaN in -> NaN out.
PM_HD double fast_atan2(double y, double x) {
    const double ax = abs_bits(x), ay = abs_bits(y);
    const bool sw = pos_gt(ay, ax);
    const double mx = sw ? ay : ax, mn = sw ? ax : ay;
    double r = atan_ratio(mn, mx);  // 0 / 0 -> NaN, replaced below
    if (sw) r = PM_T(kMisc)[1] - r;
    if (sign_bit(x)) r = PM_T(kMisc)[2] - r;
    r = with_sign_of(r, y);
    return (mx == 0.0) ? 0.0 : r;
}
// atan2(y, x) for y >= 0 and (x, y) != (0, 0): angle in [0, pi] (vector separations)
PM_HD double fast_atan2_ypos(double y, double x) {
    const double ax = abs_bits(x);
    const bool sw = pos_gt(abs_bits(y), ax);
    const double mx = sw ? y : ax, mn = sw ? ax : y;
    double r = atan_ratio(mn, mx);
    if (sw) r = PM_T(kMisc)[1] - r;
    if (sign_bit(x)) r = PM_T(kMisc)[2] - r;
    return r;
}
// atan2(y, x) for x >= 0 and (x, y) != (0, 0): angle in [-pi/2, pi/2] (latitudes)
PM_HD double fast_atan2_xpos(double y, double x) {
    const double ay = abs_bits(y);
    const bool sw = pos_gt(ay, abs_bits(x));
    const double mx = sw ? ay : x, mn = sw ? x : ay;
    double r = atan_ratio(mn, mx);
    if (sw) r = PM_T(kMisc)[1] - r;
    return with_sign_of(r, y);
}
// acos(x); NaN for |x| > 1 like the libm routine
PM_HD double fast_acos(double x) {
    return fast_atan2_ypos(fast_sqrt_nan((1.0 - x) * (1.0 + x)), x);
}

}  // namespace pm
