// pm_device.cuh - FP64 per-pixel / per-cell geometry of the PlanetMapper hot path.
//
// Each routine replaces work the reference performs with one ctypes CSPICE call per
// pixel per stage (SURVEY.md section 2, "third-party call sites") and cites the
// reference call site (file:line under /root/reference/planetmapper).  The code is
// written for the B200 FP64 pipe, not transliterated from CSPICE:
//   * everything is evaluated in the target's body frame at the reference epoch
//     t_ref = et - lt0; the per-epoch spin exp(-[omega]x dt) is applied with a
//     3-term series (|omega dt| ~ 1e-4), never with a 3x3 matrix product;
//   * the frame's J2000 vectors are rotated into that frame once per CTA
//     (FrameD), so a light-time pass is ~100 FMAs instead of ~250;
//   * the converged-Newtonian intercept runs a fixed 3 passes (the contraction
//     factor v_surface / c ~ 4e-5 makes a 4th pass a no-op in FP64) and its result
//     (point, observer, light time) is reused by the illumination and state
//     stages instead of re-solving spkcpt / illumf from scratch;
//   * angles come from atan2(|a x b|, a.b) on unnormalised vectors (same value as
//     CSPICE's vsep to 1 ulp, no normalisations, no asin);
//   * division / sqrt / trig use the MUFU-seeded routines of pm_math.cuh.
// The routines are __host__ __device__ so tests can run the identical code on the
// CPU against the oracle (tools/host_check.cu); libpm_b200.so only launches the
// __global__ kernels.
#pragma once

#include "../../include/pm_b200.h"
#include "pm_math.cuh"

namespace pm {

struct V3 {
    double x, y, z;
};

PM_HD V3 mk(double x, double y, double z) { return V3{x, y, z}; }
PM_HD V3 operator+(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
PM_HD V3 operator-(V3 a, V3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
PM_HD V3 operator-(V3 a) { return mk(-a.x, -a.y, -a.z); }
PM_HD V3 operator*(double s, V3 a) { return mk(s * a.x, s * a.y, s * a.z); }
PM_HD double dot(V3 a, V3 b) { return fma(a.x, b.x, fma(a.y, b.y, a.z * b.z)); }
PM_HD V3 cross(V3 a, V3 b) {
    return mk(fma(a.y, b.z, -a.z * b.y), fma(a.z, b.x, -a.x * b.z), fma(a.x, b.y, -a.y * b.x));
}
PM_HD V3 mul3(V3 a, const double *s) { return mk(a.x * s[0], a.y * s[1], a.z * s[2]); }
// a + s b
PM_HD V3 axpy(double s, V3 b, V3 a) { return mk(fma(s, b.x, a.x), fma(s, b.y, a.y), fma(s, b.z, a.z)); }
PM_HD double norm(V3 a) { return fast_sqrt_lite(dot(a, a)); }
PM_HD V3 ld3(const double *p) { return mk(p[0], p[1], p[2]); }
PM_HD bool finite3(V3 a) { return fabs(a.x) < INFINITY && fabs(a.y) < INFINITY && fabs(a.z) < INFINITY; }
PM_HD V3 mxv(const double *m, V3 v) {
    return mk(fma(m[0], v.x, fma(m[1], v.y, m[2] * v.z)), fma(m[3], v.x, fma(m[4], v.y, m[5] * v.z)),
              fma(m[6], v.x, fma(m[7], v.y, m[8] * v.z)));
}
PM_HD V3 mtxv(const double *m, V3 v) {
    return mk(fma(m[0], v.x, fma(m[3], v.y, m[6] * v.z)), fma(m[1], v.x, fma(m[4], v.y, m[7] * v.z)),
              fma(m[2], v.x, fma(m[5], v.y, m[8] * v.z)));
}
// Python float % 360 for finite input: inputs already in [0, 360) (every grid the map
// builders produce) return unchanged, anything else takes the exact library remainder
PM_HD_NOINLINE double pymod360_slow(double a) {
    double r = ::fmod(a, 360.0);
    if (r != 0.0 && r < 0.0) r += 360.0;
    return r;
}
PM_HD double pymod360(double a) { return (a >= 0.0 && a < 360.0) ? a : pymod360_slow(a); }

// ---------------------------------------------------------------------------------
// Frame constants + per-CTA derived values (shared memory)
// ---------------------------------------------------------------------------------
struct FrameD {
    PMFrame f;
    double inv_c;      // 1 / clight
    double inv_r[3];   // 1 / radii
    double nw[3];      // surfnm weights (min_radius / radius)^2
    double k[3];       // unit rotation axis (body frame)
    double wn;         // |omega|
    double rp;         // re (1 - f)
    double e2, ep2;    // first / second eccentricity squared of the recpgr spheroid
    double inv_omf2;   // 1 / (1 - f)^2
    double omf;        // 1 - f
    // J2000 vectors of the frame rotated into the body frame at t_ref (R0 v)
    double P0b[3], VTb[3], ATb[3], VOb[3], S0b[3], VSb[3];
    double G[9];       // R0 M^T: radrec(1, -ax, ay) vector -> ray in the body frame at t_ref
    double y0[3];      // -P0b / radii: the observer at t_ref in the scaled (unit-sphere) space of surfpt
    double y0m2;       // |y0|^2, associated as surfpt's dot(y, y)
    double As[6];      // xy -> (-ax, ay) in radians: A scaled by rpd / 3600 (first row negated)
    double inv_kmpa;   // 1 / km_per_arcsec
    int biaxial;       // intercept ellipsoid == recpgr spheroid -> closed-form geodetic
    int spin_sym;      // spheroid spinning about its symmetry axis: the image planes are taken in the t_ref frame
};

constexpr int kDeriveItems = 13;

// Exactly rounded IEEE operations for the derived constants.  The derivation runs in two places -
// in a CTA's prologue (frames read from device memory: batched launches) and on the host
// (single-frame launches, where the finished FrameD travels as a kernel parameter and the
// per-pixel code reads it as constant-bank operands) - and both must give the SAME bits, so
// nothing here may depend on MUFU seeds or on the compiler's choice of FMA contraction.
PM_HD double ex_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
PM_HD double ex_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
PM_HD double ex_div(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
PM_HD double ex_sqrt(double a) {
#ifdef __CUDA_ARCH__
    return __dsqrt_rn(a);
#else
    return ::sqrt(a);
#endif
}
// a0 b0 + a1 b1 + a2 b2 with a fixed association: (a0 b0 + a1 b1) + a2 b2, every step rounded
PM_HD double ex_dot3(double a0, double b0, double a1, double b1, double a2, double b2) {
    return ex_add(ex_add(ex_mul(a0, b0), ex_mul(a1, b1)), ex_mul(a2, b2));
}

// One independent slice of the derived constants (one thread of a CTA, or a host loop).
PM_HD void derive_frame_item(FrameD &s, int item) {
    const PMFrame &f = s.f;
    if (item >= 3 && item <= 8) {
        const double *src = item == 3 ? f.P0 : item == 4 ? f.VT : item == 5 ? f.AT : item == 6 ? f.VO : item == 7 ? f.S0 : f.VS;
        double *dst = item == 3 ? s.P0b : item == 4 ? s.VTb : item == 5 ? s.ATb : item == 6 ? s.VOb : item == 7 ? s.S0b : s.VSb;
        for (int r = 0; r < 3; r++)
            dst[r] = ex_dot3(f.R0[3 * r], src[0], f.R0[3 * r + 1], src[1], f.R0[3 * r + 2], src[2]);
        if (item == 3) {
            // the first light-time pass of sincpt starts every pixel's ray at this observer: its scaled
            // position and |.|^2 with the same roundings as surfpt's mul3(o, inv_r) and dot(y, y)
            for (int r = 0; r < 3; r++) s.y0[r] = ex_mul(-dst[r], ex_div(1.0, f.radii[r]));
            s.y0m2 = fma(s.y0[0], s.y0[0], fma(s.y0[1], s.y0[1], ex_mul(s.y0[2], s.y0[2])));
        }
    } else if (item >= 9 && item <= 11) {
        const int r = item - 9;  // row r of R0 M^T
        for (int c = 0; c < 3; c++)
            s.G[3 * r + c] = ex_dot3(f.R0[3 * r], f.M[3 * c], f.R0[3 * r + 1], f.M[3 * c + 1], f.R0[3 * r + 2], f.M[3 * c + 2]);
    } else if (item == 12) {
        const double sc = kRpd / 3600.0;
        for (int c = 0; c < 3; c++) {
            s.As[c] = -ex_mul(f.A[c], sc);
            s.As[3 + c] = ex_mul(f.A[3 + c], sc);
        }
        s.inv_kmpa = ex_div(1.0, f.km_per_arcsec);
    } else if (item == 0) {
        s.inv_c = ex_div(1.0, f.clight);
        const double w2 = ex_dot3(f.omega[0], f.omega[0], f.omega[1], f.omega[1], f.omega[2], f.omega[2]);
        const double wn = ex_sqrt(w2);
        s.wn = wn;
        s.k[0] = wn > 0.0 ? ex_div(f.omega[0], wn) : 0.0;
        s.k[1] = wn > 0.0 ? ex_div(f.omega[1], wn) : 0.0;
        s.k[2] = wn > 0.0 ? ex_div(f.omega[2], wn) : 0.0;
        // A spin about the z axis commutes with the scaling of a spheroid with radii[0] == radii[1], so the
        // intercept and the illumination angles can be solved in the t_ref frame (image_pixel<kSpinSym>).
        // What that neglects is the spin axis' tilt off z: a displacement of at most |omega_perp| dt (a - c)
        // of the surface, with |dt| <= 2 a / clight over the disc.  Allowed up to 1e-9 km, far below the
        // ~4e-7 km that one ulp of the epoch et - lt moves the target (DESIGN.md section 5); 0 for a sphere.
        const double wperp = ex_sqrt(ex_add(ex_mul(f.omega[0], f.omega[0]), ex_mul(f.omega[1], f.omega[1])));
        const double flat = fabs(ex_add(f.radii[0], -f.radii[2]));
        const double shift = ex_mul(ex_mul(wperp, ex_div(ex_mul(2.0, f.radii[0]), f.clight)), flat);
        s.spin_sym = (f.radii[0] == f.radii[1]) && (shift <= 1.0e-9);
    } else if (item == 1) {
        const double a = f.radii[0], b = f.radii[1], c = f.radii[2];
        s.inv_r[0] = ex_div(1.0, a);
        s.inv_r[1] = ex_div(1.0, b);
        s.inv_r[2] = ex_div(1.0, c);
        const double m = fmin(a, fmin(b, c));
        const double ma = ex_div(m, a), mb = ex_div(m, b), mc = ex_div(m, c);
        s.nw[0] = ex_mul(ma, ma);
        s.nw[1] = ex_mul(mb, mb);
        s.nw[2] = ex_mul(mc, mc);
    } else if (item == 2) {
        const double rp = ex_add(f.re, -ex_mul(f.f, f.re));
        const double re2 = ex_mul(f.re, f.re), rp2 = ex_mul(rp, rp);
        const double omf = ex_add(1.0, -f.f);
        s.rp = rp;
        s.e2 = ex_add(1.0, -ex_div(rp2, re2));
        s.ep2 = ex_add(ex_div(re2, rp2), -1.0);
        s.omf = omf;
        s.inv_omf2 = ex_div(1.0, ex_mul(omf, omf));
        s.biaxial = (f.radii[0] == f.radii[1]) && (f.re == f.radii[0]) && (fabs(rp - f.radii[2]) <= 4e-16 * f.radii[2]);
    }
}

#ifdef __CUDACC__
// Cooperative load of one PMFrame into shared memory + derived constants.  The
// derivation is spread over the four warps of the CTA so that items with different
// code paths run concurrently instead of serialising inside one warp:
// warp 0: the six R0 v products, warp 1: R0 M^T rows + pixel affine, warp 2: spin /
// radii reciprocals, warp 3: spheroid constants.
__device__ __forceinline__ void load_frame(FrameD &s, const PMFrame *__restrict__ g) {
    const double *src = reinterpret_cast<const double *>(g);
    double *dst = reinterpret_cast<double *>(&s.f);
    for (int i = threadIdx.x; i < PM_FRAME_NDOUBLES; i += blockDim.x) dst[i] = __ldg(src + i);
    __syncthreads();
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    int item = -1;
    if (blockDim.x >= 128) {
        if (w == 0 && l < 6) item = 3 + l;
        else if (w == 1 && l < 4) item = 9 + l;
        else if (w == 2 && l < 2) item = l;
        else if (w == 3 && l == 0) item = 2;
    } else if (threadIdx.x < kDeriveItems) {
        item = threadIdx.x;
    }
    if (item >= 0) derive_frame_item(s, item);
    __syncthreads();
}
#endif
inline void load_frame_host(FrameD &s, const PMFrame *g) {
    s.f = *g;
    for (int i = 0; i < kDeriveItems; i++) derive_frame_item(s, i);
}

// cos^2 (scaled-space emission) below which sincpt iterates to convergence: emission > ~86.9 deg.
// Above it the fixed-point step's own error (the light time is not linear in the epoch:
// V^3 de^2 / (2 r c^2 cos^4 e) km) stays below the target motion in one epoch quantum ulp(et) ~ 3e-8 s
// (V ulp(et) / cos e), which is the resolution of CSPICE's own result.
#ifndef PM_GRAZING_COS2
#define PM_GRAZING_COS2 3.0e-3
#endif
constexpr double kGrazingCos2 = PM_GRAZING_COS2;

// Per-pixel literals that are not exact in a DADD / DFMA immediate, in pairs used together (one 16-byte
// constant load each instead of two 32-bit moves per literal); the spin series reads kTinyC (pm_math.cuh)
enum PixC {
    kPixDt1Min = 0,   // sincpt: |dt1| above which the two-pass fixed point is used
    kPixGrazing = 1,  // sincpt: kGrazingCos2
    kPixInv60 = 2,    // local_solar_time: 1/60, 1/3600
    kPixInv3600 = 3,
    kPixRpd = 4,      // local_solar_time: rad per deg
    kPixBetaMax = 5,  // doppler_factor / radial_velocity: |v| / c bound of the series
};
PM_DEV_TABLE(kPixC, 6, 1.0e-6, kGrazingCos2, 1.0 / 60.0, 1.0 / 3600.0, kRpd, 1.0e-3)

// ---------------------------------------------------------------------------------
// Frame spin: body frame at t_ref  <->  body frame at t_ref + dt
// ---------------------------------------------------------------------------------
// sin(theta), 1 - cos(theta) for theta = |omega| dt
struct Rot {
    double s, omc;
};
PM_HD Rot make_rot(const FrameD &fs, double dt) {
    const double th = fs.wn * dt;
    Rot r;
    if (fabs(th) < 0.001953125) {  // 2^-9: series exact to < 1e-20 relative
        const double z = th * th;
        r.s = th * fma(z, fma(z, PM_T(kTinyC)[0], PM_T(kTinyC)[2]), 1.0);  // 1/120, -1/6
        r.omc = z * fma(z, fma(z, -PM_T(kTinyC)[1], -PM_T(kTinyC)[3]), 0.5);  // 1/720, -1/24
    } else {
        double sh, ch;
        sincos_lib(0.5 * th, &sh, &ch);
        r.s = 2.0 * sh * ch;
        r.omc = 2.0 * sh * sh;
    }
    return r;
}
// exp(-theta [k]x) w = w + sin(theta) (w x k) + (1 - cos(theta)) (k (k.w) - w)
PM_HD V3 spin_fwd(const FrameD &fs, Rot r, V3 w) {
    const V3 k = ld3(fs.k);
    const V3 c = cross(w, k);
    const double kw = dot(k, w);
    const V3 t = mk(fma(k.x, kw, -w.x), fma(k.y, kw, -w.y), fma(k.z, kw, -w.z));
    return axpy(r.omc, t, axpy(r.s, c, w));
}
// exp(+theta [k]x) u (inverse spin); kxu = k x u may be supplied by the caller
PM_HD V3 spin_bwd_c(const FrameD &fs, Rot r, V3 u, V3 kxu) {
    const V3 k = ld3(fs.k);
    const double ku = dot(k, u);
    const V3 t = mk(fma(k.x, ku, -u.x), fma(k.y, ku, -u.y), fma(k.z, ku, -u.z));
    return axpy(r.omc, t, axpy(r.s, kxu, u));
}
PM_HD V3 spin_bwd(const FrameD &fs, Rot r, V3 u) { return spin_bwd_c(fs, r, u, cross(ld3(fs.k), u)); }
// pxform('J2000', body, t_ref + dt) v   (inside sincpt / illumf / spkcpt, body.py:998)
PM_HD V3 to_body(const FrameD &fs, Rot r, V3 v) { return spin_fwd(fs, r, mxv(fs.f.R0, v)); }
// pxform(body, 'J2000', t_ref + dt) u   (body.py:940)
PM_HD V3 from_body(const FrameD &fs, Rot r, V3 u) { return mtxv(fs.f.R0, spin_bwd(fs, r, u)); }
// target centre relative to the observer at t_ref + dt, in the body frame at t_ref
PM_HD V3 target_pos_b(const FrameD &fs, double dt) {
    const double h = 0.5 * dt * dt;
    return mk(fma(fs.ATb[0], h, fma(fs.VTb[0], dt, fs.P0b[0])), fma(fs.ATb[1], h, fma(fs.VTb[1], dt, fs.P0b[1])),
              fma(fs.ATb[2], h, fma(fs.VTb[2], dt, fs.P0b[2])));
}

// ---------------------------------------------------------------------------------
// Angles
// ---------------------------------------------------------------------------------
// spice.recrad angles (base.py:902): RA in [0, 2pi), Dec
PM_HD void recrad_angles(V3 v, double &ra, double &dec) {
    dec = fast_atan2_xpos(v.z, fast_sqrt(fma(v.x, v.x, v.y * v.y)));
    double lon = fast_atan2(v.y, v.x);
    if (lon < 0.0) lon += kTwoPi;
    ra = lon;
}
// spice.radrec(1, ra, dec) (body.py:967, :1369), any finite angles
PM_HD V3 radrec1(double ra, double dec) {
    double sr, cr, sd, cd;
    sincos_full(ra, sr, cr);
    sincos_full(dec, sd, cd);
    return mk(cr * cd, sr * cd, sd);
}
// spice.vsep for any two non-zero vectors: atan2(|a x b|, a.b)
PM_HD double vsep(V3 a, V3 b) { return fast_atan2_ypos(norm(cross(a, b)), dot(a, b)); }

// spice.surfpt (inside sincpt, body.py:1010): nearest ray / ellipsoid intersection,
// perpendicular-projection form.  o, u in the body frame; p = o + t u.
struct RayHit {
    V3 pp;        // foot of the perpendicular from the centre to the ray, scaled (unit-sphere) space
    double ixx;   // 1 / |x|^2, x = u / radii
    double a;     // ray parameter of that foot: pp = y + a x (for a unit u: km from the observer)
    double t;     // ray parameter of the intercept, t = a - h with the half-chord h = sqrt((1 - |pp|^2) ixx)
    double cos2;  // 1 - |pp|^2: squared half-chord in the unit-sphere space, -> 0 at tangency
};
// y: the ray's origin in the scaled (unit-sphere) space, ym2 = |y|^2 (surfpt below, or per frame);
// x = u / radii: the ray's direction in that space, ixx = 1 / |x|^2
PM_HD bool surfpt_yx(const FrameD &fs, V3 y, double ym2, V3 x, double ixx, V3 &p, RayHit &hit) {
    const double yx = dot(y, x);
    const double a = -(yx * ixx);
    const V3 pp = axpy(a, x, y);  // component of y perpendicular to the ray
    const double pm2 = dot(pp, pp);
    if (!(pm2 < INFINITY)) return false;
    hit.pp = pp;
    hit.ixx = ixx;
    hit.a = a;
    hit.cos2 = 1.0 - pm2;
    double h;
    if (ym2 > 1.0) {
        if (pm2 > 1.0) return false;
        if (yx > 0.0) return false;
        h = -fast_sqrt_lite((1.0 - pm2) * ixx);
    } else if (ym2 == 1.0) {
        h = -a;  // the origin itself
    } else {
        h = fast_sqrt_lite(fmax(0.0, 1.0 - pm2) * ixx);
    }
    hit.t = a + h;
    p = mul3(axpy(h, x, pp), fs.f.radii);
    return true;
}
PM_HD bool surfpt_y(const FrameD &fs, V3 y, double ym2, V3 u, V3 &p, RayHit &hit) {
    // scaled space (unit sphere); the direction x is deliberately NOT normalised: the
    // three dot products are independent and a single reciprocal serves both the
    // projection and the half-chord
    const V3 x = mul3(u, fs.inv_r);
    const double xx = dot(x, x);
    if (!(xx > 0.0)) return false;
    return surfpt_yx(fs, y, ym2, x, fast_rcp(xx), p, hit);
}
PM_HD bool surfpt(const FrameD &fs, V3 o, V3 u, V3 &p, RayHit &hit) {
    const V3 y = mul3(o, fs.inv_r);
    return surfpt_y(fs, y, dot(y, y), u, p, hit);
}

// Result of the converged intercept, everything in the body frame at the intercept
// epoch t_ref + dt unless stated.
struct Intercept {
    V3 p;        // surface point (body-fixed)
    V3 u;        // unit ray observer -> point in the body frame at the intercept epoch: the line of sight
                 // itself (exact), not (p - o) / L, which carries p's error magnified by r / L for a near observer
                 // (general path only)
    V3 p0;       // the surface point in the body frame at t_ref (spin-symmetric path only)
    Rot r;       // spin over dt
    double dt;   // intercept epoch - t_ref
    double L;    // observer -> point range (km)
    double lt;   // L / c
};

// Slow path of sincpt for grazing rays and for frames whose first two passes coincide in
// epoch: CSPICE's loop as written - full intercepts until the FP64 epoch et - lt stops
// changing (at most 10 passes in total).  dt (in: epoch offset of the next pass) and p come
// back for the converged pass.  Kept out of line so the common path keeps its registers.
// kSpinSym (FrameD::spin_sym): every pass is solved in the body frame at t_ref, so p is the point in that frame.
template <bool kSpinSym>
PM_HD_NOINLINE bool sincpt_converge(const FrameD &fs, V3 u0, double &dt, V3 &p, double &range) {
    const PMFrame &f = fs.f;
    for (int it = 0; it < 8; it++) {
        V3 o = -target_pos_b(fs, dt), u = u0;
        if (!kSpinSym) {
            const Rot r = make_rot(fs, dt);
            o = spin_fwd(fs, r, o);
            u = spin_fwd(fs, r, u0);
        }
        RayHit hit;
        if (!surfpt(fs, o, u, p, hit)) return false;
        range = hit.t;
        const double t = dt + f.t_ref;
        const double t_new = f.et - hit.t * fs.inv_c;  // u0 is a unit vector: the ray parameter is the range
        if (!(fabs(t_new - t) > 1.0e-17 * fabs(t_new))) break;
        dt = t_new - f.t_ref;
    }
    return true;
}

// spice.sincpt(..., 'CN', ..., d) (body.py:1008-1020): intercept with the light time
// iterated on the intercept point.  u0: UNIT ray direction in the body frame at t_ref (ray parameters
// are used as ranges).
//
// CSPICE iterates  epoch e_{i+1} = et - lt(e_i)  from e_0 = et - lt0 = t_ref until the
// light time stops changing; the epochs contract geometrically with ratio V_lateral tan(emission) / c
// (4e-5 at the disc centre, 5e-3 at 89 deg).  Here
//   pass 1 (e_0): dt = 0, the spin is the identity (exactly CSPICE's first pass);
//   pass 2 (e_1): full intercept;
//   then the fixed point e* of the loop is taken from the ratio of the two steps, and the intercept at
//   e* is assembled from quantities of the two solves that ARE smooth in the epoch (see below) - no
//   third ray / ellipsoid solve.  The ranges are the ray parameters themselves (u0 is a unit vector).
//   Grazing rays (cos^2 of the scaled-space emission <= kGrazingCos2, i.e. emission > ~86.9 deg) are the
//   exception: there the light time is too far from linear in the epoch for the two-point fixed point,
//   so those pixels run CSPICE's loop as written (until et - lt is stable).
//
// kSpinSym (FrameD::spin_sym): the body is a spheroid spinning about its symmetry axis.  Spinning the
// observer and the ray together about that axis leaves the ray / ellipsoid solve unchanged, so every pass
// is solved in the body frame at t_ref - observer -target_pos_b(dt), ray u0 - and only the final point is
// spun to its epoch.  Pass 2 then shares pass 1's direction x and 1 / |x|^2, and it.p0 holds the point at
// t_ref; it.u is not set.
template <bool kSpinSym = false>
PM_HD bool sincpt(const FrameD &fs, V3 u0, Intercept &it) {
    const PMFrame &f = fs.f;
    V3 p1, p2;
    RayHit h1, h2;
    const V3 x = mul3(u0, fs.inv_r);
    const double xx = dot(x, x);
    if (!(xx > 0.0)) return false;
    const double ixx = fast_rcp(xx);
    if (!surfpt_yx(fs, ld3(fs.y0), fs.y0m2, x, ixx, p1, h1)) return false;  // observer at t_ref: -P0b
    const double lt1 = h1.t * fs.inv_c;  // u0 is a unit vector: the ray parameter is the range

    const double dt1 = (f.et - lt1) - f.t_ref;
    if (kSpinSym) {
        const V3 y2 = mul3(-target_pos_b(fs, dt1), fs.inv_r);
        if (!surfpt_yx(fs, y2, dot(y2, y2), x, ixx, p2, h2)) return false;
    } else {
        const Rot r1 = make_rot(fs, dt1);
        if (!surfpt(fs, spin_fwd(fs, r1, -target_pos_b(fs, dt1)), spin_fwd(fs, r1, u0), p2, h2)) return false;
    }
    const double lt2 = h2.t * fs.inv_c;

    // epochs as CSPICE forms them: et - lt rounded to a double (granularity ulp(et) ~ 3e-8 s,
    // i.e. ~1e-6 km of target motion)
    double dt = (f.et - lt2) - f.t_ref;
    V3 p;
    double L;
    if (fabs(dt1) > PM_T(kPixC)[kPixDt1Min] && h2.cos2 > PM_T(kPixC)[kPixGrazing]) {
        // The epochs e_0 = t_ref, e_1, e_2 of CSPICE's loop contract geometrically (ratio (e_2 - e_1) /
        // (e_1 - e_0)); the loop's fixed point is e_1 + lam (e_1 - e_0), lam = (e_2 - e_1) / (e_1 - e_2 + e_1 - e_0).
        // The intercept there comes from the two solves without a third one: the foot pp of the
        // perpendicular from the centre to the ray, its ray parameter a (an inertial quantity: linear in
        // the epoch up to the target's acceleration) and 1 / |x|^2 are smooth in the epoch and are moved along
        // their secants, the ray direction is spun to the new epoch exactly, and the half-chord
        // h = sqrt((1 - |pp|^2) / |x|^2) - the one ingredient that is NOT smooth towards the limb - is formed
        // from them.  (Moving the intercept itself along its secant leaves an error ~ 1 / cos^3(emission):
        // invisible under the |P0| rounding of a distant observer, 1.6e-7 deg at 88 deg emission from 2.5 radii.)
        const double lam = fast_div_lite(dt - dt1, dt1 - (dt - dt1));
        dt = fma(lam, dt1, dt1) + f.t_ref;  // the fixed point, rounded as et - lt is
        dt -= f.t_ref;
        const V3 pps = axpy(lam, h2.pp - h1.pp, h2.pp);
        const double ixxs = kSpinSym ? ixx : fma(lam, h2.ixx - h1.ixx, h2.ixx);
        const double hs = fast_sqrt_lite(fmax(1.0 - dot(pps, pps), 0.0) * ixxs);
        L = fma(lam, h2.a - h1.a, h2.a) - hs;
        it.r = make_rot(fs, dt);
        if (kSpinSym) {
            it.p0 = axpy(-hs, u0, mul3(pps, fs.f.radii));
            p = spin_fwd(fs, it.r, it.p0);
        } else {
            it.u = spin_fwd(fs, it.r, u0);
            p = axpy(-hs, it.u, mul3(pps, fs.f.radii));
        }
    } else {
        double dt_c = dt, L_c;  // address-taken copies: keep dt and p themselves in registers
        V3 p_c;
        if (!sincpt_converge<kSpinSym>(fs, u0, dt_c, p_c, L_c)) return false;
        dt = dt_c;
        L = L_c;
        it.r = make_rot(fs, dt);
        if (kSpinSym) {
            it.p0 = p_c;
            p = spin_fwd(fs, it.r, p_c);
        } else {
            p = p_c;
            it.u = spin_fwd(fs, it.r, u0);
        }
    }
    it.p = p;
    it.dt = dt;
    it.L = L;
    it.lt = L * fs.inv_c;
    return true;
}

// Geodetic latitude / altitude of an arbitrary point w.r.t. the spheroid
// (re, re, re(1-f)): spice.recgeo inside spice.recpgr (body.py:1030, :2592).
// Bowring's iteration on the (sin, cos) of the reduced latitude - no trig calls, no
// division, well defined at the poles.
PM_HD void geodetic_general(const FrameD &fs, double rho, double z, double &lat, double &alt) {
    const PMFrame &f = fs.f;
    if (f.f == 0.0) {
        lat = fast_atan2_xpos(z, rho);
        alt = fast_sqrt(fma(rho, rho, z * z)) - f.re;
        return;
    }
    // reduced latitude beta: tan(beta) = re z / (rp rho)
    double sb = f.re * z, cb = fs.rp * rho;
    double n = fast_rsqrt(fma(sb, sb, cb * cb) + sqrt_guard());
    sb *= n;
    cb *= n;
    double num = z, den = rho;
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        num = fma(fs.ep2 * fs.rp, sb * sb * sb, z);
        den = fma(-fs.e2 * f.re, cb * cb * cb, rho);
        double nsb = fs.omf * num, ncb = den;
        n = fast_rsqrt(fma(nsb, nsb, ncb * ncb) + sqrt_guard());
        nsb *= n;
        ncb *= n;
        const double change = fabs(nsb - sb) + fabs(ncb - cb);
        sb = nsb;
        cb = ncb;
        if (change <= 4.0e-16) break;
    }
    lat = fast_atan2(num, den);
    n = fast_rsqrt(fma(num, num, den * den) + sqrt_guard());
    const double sp = num * n, cp = den * n;
    alt = fma(rho, cp, z * sp) - f.re * fast_sqrt(fma(-fs.e2 * sp, sp, 1.0));
}

// Geodetic latitude w.r.t. an arbitrary spheroid (re, re, rp): the same iteration with the
// constants derived on the spot.  Only used by the point transforms (planetocentric inputs
// combined with an altitude), never per pixel.
PM_HD double geodetic_lat_spheroid(double re, double rp, double rho, double z) {
    if (re == rp) return fast_atan2_xpos(z, rho);
    const double q = fast_div(rp, re), qi = fast_div(re, rp);
    const double e2 = fma(-q, q, 1.0), ep2 = fma(qi, qi, -1.0);
    double sb = re * z, cb = rp * rho;
    double n = fast_rsqrt(fma(sb, sb, cb * cb) + sqrt_guard());
    sb *= n;
    cb *= n;
    double num = z, den = rho;
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        num = fma(ep2 * rp, sb * sb * sb, z);
        den = fma(-e2 * re, cb * cb * cb, rho);
        double nsb = q * num, ncb = den;
        n = fast_rsqrt(fma(nsb, nsb, ncb * ncb) + sqrt_guard());
        nsb *= n;
        ncb *= n;
        const double change = fabs(nsb - sb) + fabs(ncb - cb);
        sb = nsb;
        cb = ncb;
        if (change <= 4.0e-16) break;
    }
    return fast_atan2(num, den);
}

// spice.recpgr (body.py:1030): planetographic lon in [0, 2pi), lat, alt
PM_HD void recpgr(const FrameD &fs, V3 p, bool on_spheroid, double &lon, double &lat, double &alt) {
    const double rho = fast_sqrt(fma(p.x, p.x, p.y * p.y));
    double l = fs.f.lon_sign * fast_atan2(p.y, p.x);
    if (l < 0.0) l += kTwoPi;
    lon = l;
    if (on_spheroid) {
        // the point lies on the spheroid itself: its normal is the geodetic normal
        lat = fast_atan2_xpos(p.z * fs.inv_omf2, rho);
        alt = 0.0;
    } else {
        geodetic_general(fs, rho, p.z, lat, alt);
    }
}

// spice.pgrrec(lon, lat, alt = 0) (body.py:903), radians in
PM_HD V3 pgrrec0(const FrameD &fs, double lon, double lat) {
    const PMFrame &f = fs.f;
    double slat, clat, slon, clon;
    sincos_full(lat, slat, clat);
    sincos_full(f.lon_sign * lon, slon, clon);
    const double x = f.re * clat, y = fs.rp * slat;
    const double scale = fast_rsqrt(fma(x, x, y * y) + sqrt_guard());
    return mk(scale * clon * x * f.re, scale * slon * x * f.re, scale * y * fs.rp);
}

// spice.reclat angles (body.py:2912)
PM_HD void reclat_angles(V3 v, double &lon, double &lat) {
    lat = fast_atan2_xpos(v.z, fast_sqrt(fma(v.x, v.x, v.y * v.y)));
    lon = fast_atan2(v.y, v.x);
}

// Body.local_solar_time_from_lon (body.py:2364-2398) -> spice.et2lst 'planetographic'
// lon_deg finite.  Whole seconds are split with integer arithmetic; the two divisions
// of the reference's `hr + mn / 60 + sc / 3600` are reproduced correctly rounded.
PM_HD double local_solar_time(const PMFrame &f, double lon_deg) {
    double ang = f.lon_sign * (lon_deg * PM_T(kPixC)[kPixRpd]) - f.sun_lon_lst;
    if (f.prograde == 0.0) ang = -ang;
    // fmod(ang, 2 pi) folded into [0, 2 pi): ang - k 2pi is exact for the small k here
    const double k = floor(ang * PM_T(kMisc)[8]);
    ang = fma(-k, PM_T(kMisc)[7], ang);
    if (ang < 0.0) ang += PM_T(kMisc)[7];
    if (ang >= PM_T(kMisc)[7]) ang -= PM_T(kMisc)[7];
    double sec = fma(ang, 86400.0 / kTwoPi, 43200.0);
    if (sec >= 86400.0) sec -= 86400.0;
    const int isec = (int)sec;  // floor: sec >= 0
    const int hr = isec / 3600, rem = isec - hr * 3600;
    const int mn = rem / 60, sc = rem - mn * 60;
    // correctly rounded mn / 60 and sc / 3600 (Markstein: r = RN(1/b), one FMA correction)
    const double dm = (double)mn, ds = (double)sc;
    double qm = dm * PM_T(kPixC)[kPixInv60];
    qm = fma(fma(-60.0, qm, dm), PM_T(kPixC)[kPixInv60], qm);
    double qs = ds * PM_T(kPixC)[kPixInv3600];
    qs = fma(fma(-3600.0, qs, ds), PM_T(kPixC)[kPixInv3600], qs);
    return ((double)hr + qm) + qs;
}

// SpiceBase.calculate_doppler_factor (base.py:524-551)
// the closed forms, for |v| >= 1e-3 c: out of line so that the per-pixel code does not carry (or if-convert) them
PM_HD_NOINLINE double doppler_factor_closed(double beta) { return fast_sqrt(fast_div(1.0 + beta, 1.0 - beta)); }
PM_HD_NOINLINE double light_time_rate_closed(double a, double b, double c) { return fast_div(a - b, c + a); }
PM_HD double doppler_factor(const FrameD &fs, double rv) {
    const double beta = rv * fs.inv_c;
    // sqrt((1 + b) / (1 - b)) = (1 + b) (1 - b^2)^(-1/2) = 1 + b + b^2/2 + b^3/2 + 3 b^4/8 + 3 b^5/8 + 5 b^6/16 + ...
    // For |b| < 1e-3 (300 km/s; solar-system radial velocities are < 1e-4 c) the first omitted term is
    // < 3.2e-19: the sum is within one ulp of the correctly rounded quotient and root, without either.
    if (fabs(beta) < PM_T(kPixC)[kPixBetaMax])
        return fma(beta, fma(beta, fma(beta, fma(beta, fma(beta, 0.375, 0.375), 0.5), 0.5), 1.0), 1.0);
    return doppler_factor_closed(beta);
}

// radial velocity of spkcpt's state (body.py:2830-2853) from projections on the unit
// line of sight: a = V_point . ph, b = V_observer . ph
PM_HD double radial_velocity(const FrameD &fs, double a, double b) {
    // d(light time)/dt = (a - b) / (c + a).  It only scales a ~1e-4 correction of the result, so
    // 1 / (c + a) = (1 - a/c + (a/c)^2 - ...) / c is cut after the square (relative error (a/c)^3 < 1e-9
    // of the correction for |a| < 300 km/s)
    const double ac = a * fs.inv_c;
    double dlt = (a - b) * fs.inv_c * fma(ac, ac - 1.0, 1.0);
    if (!(fabs(ac) < PM_T(kPixC)[kPixBetaMax])) dlt = light_time_rate_closed(a, b, fs.f.clight);
    return fma(-dlt, a, a) - b;
}

struct Illum {
    double phase, incdnc, emissn, azimuth;  // radians
};
// spice.illumf angles (body.py:1915-1935) + Body._azimuth_angle_from_gie_radians
// (body.py:2319-2332) from three body-frame vectors at the point epoch:
// n surface normal, s point -> Sun, e point -> observer (any magnitudes).
PM_HD void illum_angles(V3 n, V3 s, V3 e, bool want_az, Illum &out) {
    const V3 cse = cross(s, e), cns = cross(n, s), cne = cross(n, e);
    const double dse = dot(s, e), dns = dot(n, s), dne = dot(n, e);
    const double mns = norm(cns), mne = norm(cne);
    out.phase = fast_atan2_ypos(norm(cse), dse);
    out.incdnc = fast_atan2_ypos(mns, dns);
    out.emissn = fast_atan2_ypos(mne, dne);
    if (want_az) {
        // pi - acos of (cos g - cos e cos i) / (sin e sin i), i.e. of the cosine of the angle between
        // n x e and n x s, written as the atan2 of that angle's sine and cosine: by Lagrange's identity
        // (n x e).(n x s) = (s.e)(n.n) - (n.e)(n.s) and |(n x e) x (n x s)| = |n| |n.(s x e)|.  No division
        // or acos, and well conditioned where sin e or sin i -> 0 (acos of a 0 / 0 quotient there)
        const double nn = dot(n, n);
        const double a = fma(dse, nn, -dne * dns);
        out.azimuth = fast_atan2_ypos(fast_sqrt_pos(nn) * fabs(dot(n, cse)), -a);  // pi - atan2(y, a)
    }
}

// Point -> Sun vector of the point p0 (body frame at t_ref) at epoch offset dt, in the body
// frame at t_ref.  Solves the Sun -> point light time from the frame's seed lts0.  VS is the
// Sun's barycentric velocity (~0.013 km/s): the contraction factor of the iteration is
// VS / c ~ 4e-8 and the seed is off by <= R / c, so ONE refinement leaves a Sun-direction
// error below 1e-18 rad.
PM_HD V3 sun_vec0(const FrameD &fs, V3 p0, double dt) {
    const PMFrame &f = fs.f;
    const double h = 0.5 * dt * dt;
    // target-centre displacement since t_ref + point offset, body frame at t_ref
    const V3 base = mk(fs.S0b[0] - fma(fs.ATb[0], h, fma(fs.VTb[0], dt, p0.x)),
                       fs.S0b[1] - fma(fs.ATb[1], h, fma(fs.VTb[1], dt, p0.y)),
                       fs.S0b[2] - fma(fs.ATb[2], h, fma(fs.VTb[2], dt, p0.z)));
    const V3 VSb = ld3(fs.VSb);
    const V3 sv = axpy(dt, VSb, base);
    const double lts = fast_sqrt_pos(dot(sv, sv)) * fs.inv_c;  // the Sun is never at the point
    return axpy(dt - (lts - f.lts0), VSb, base);
}
// Illumination geometry of body-fixed point p at epoch offset dt (spin r), given the
// point -> observer vector e (body frame at the epoch).
PM_HD void illum_at(const FrameD &fs, V3 p, V3 p0 /* spin_bwd(p) */, V3 e, Rot r, double dt, bool want_az,
                    Illum &out) {
    const V3 s_b = spin_fwd(fs, r, sun_vec0(fs, p0, dt));
    const V3 n = mul3(p, fs.nw);  // spice.surfnm direction
    illum_angles(n, s_b, e, want_az, out);
}

// Converged apparent geometry of a body-fixed point (spice.spkcpt, body.py:2830-2845;
// the light-time half of spice.illumf, body.py:1915-1935).
struct PointGeom {
    V3 p0;       // spin_bwd(p): point in the body frame at t_ref
    V3 X0;       // observer -> point, body frame at t_ref
    Rot r;
    double dt, L, lt;
};
PM_HD void point_geom(const FrameD &fs, V3 p, PointGeom &g) {
    const PMFrame &f = fs.f;
    // pass 1 at dt = 0 (identity spin)
    double lt = norm(ld3(fs.P0b) + p) * fs.inv_c;
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
        const double dt = (f.et - lt) - f.t_ref;
        const Rot r = make_rot(fs, dt);
        const V3 p0 = spin_bwd(fs, r, p);
        const V3 X0 = target_pos_b(fs, dt) + p0;
        const double L = norm(X0);
        lt = L * fs.inv_c;
        g.p0 = p0;
        g.X0 = X0;
        g.r = r;
        g.dt = dt;
        g.L = L;
        g.lt = lt;
    }
}
// radial velocity for a point with geometry g (body-fixed point p)
PM_HD double point_rv(const FrameD &fs, V3 p, const PointGeom &g) {
    const double iL = fast_rcp(g.L);
    const V3 ph0 = iL * g.X0;
    const V3 vt = axpy(g.dt, ld3(fs.ATb), ld3(fs.VTb));
    // (omega x p) . ph in the epoch frame = (omega x p) . spin_fwd(X0) / L; the rotation
    // commutes with the dot product, so use spin_bwd on the velocity side instead:
    const V3 vrot0 = spin_bwd(fs, g.r, cross(ld3(fs.f.omega), p));
    const double a = dot(vt + vrot0, ph0);
    const double b = dot(ld3(fs.VOb), ph0);
    return radial_velocity(fs, a, b);
}

// Body._azimuth_angle_from_gie_radians for the oracle-style call sites
PM_HD V3 xy2ray_local(const FrameD &fs, double x, double y) {
    // BodyXY._xy2obsvec_norm (body_xy.py:375-377) + Body._angular2obsvec_norm
    // (body.py:1363-1373): radrec(1, -ax, ay) with ax, ay from the affine map
    const double ra = fma(fs.As[0], x, fma(fs.As[1], y, fs.As[2]));
    const double dec = fma(fs.As[3], x, fma(fs.As[4], y, fs.As[5]));
    double sr, cr, sd, cd;
    sincos_small2(ra, dec, sr, cr, sd, cd);
    return mk(cr * cd, sr * cd, sd);
}

// Body._obsvec2angular (body.py:1345-1361), arcsec; ov finite
PM_HD void obsvec2angular(const PMFrame &f, V3 ov, double &ax, double &ay) {
    double ra, dec;
    recrad_angles(mxv(f.M, ov), ra, dec);
    double x = pymod360(-(ra * kDpr));
    if (x > 180.0) x -= 360.0;
    ax = x * 3600.0;
    ay = (dec * kDpr) * 3600.0;
}

// Body._targvec2obsvec (body.py:917-948)
PM_HD V3 targvec2obsvec(const FrameD &fs, V3 tv) {
    const PMFrame &f = fs.f;
    const V3 off = tv - ld3(f.sub_t);
    const double dist_offset = norm(ld3(f.sub_ray) + off) - f.sub_dist;
    const double sub_et = f.t_ref + f.sub_dt;
    const double tt = sub_et - dist_offset * fs.inv_c;
    const Rot r = make_rot(fs, tt - f.t_ref);
    return ld3(f.sub_obs) + from_body(fs, r, off);
}

// Body._obsvec2targvec (body.py:972-1006), including its frame-mixing norm
PM_HD V3 obsvec2targvec(const FrameD &fs, V3 ov) {
    const PMFrame &f = fs.f;
    const V3 off = ov - ld3(f.sub_obs);
    const double dist_offset = norm(off - ld3(f.sub_ray)) - f.sub_dist;
    const double sub_et = f.t_ref + f.sub_dt;
    const double tt = sub_et - dist_offset * fs.inv_c;
    const Rot r = make_rot(fs, tt - f.t_ref);
    return ld3(f.sub_t) + to_body(fs, r, off);
}

// Body._ring_coordinates_from_obsvec(only_visible=False) (body.py:2577-2615); ov finite
PM_HD void ring_coordinates(const FrameD &fs, V3 ov, double &radius, double &lon_deg, double &dist) {
    const PMFrame &f = fs.f;
    radius = lon_deg = dist = NAN;
    const double nd = dot(ld3(f.ring_n), ov);  // spice.inrypl, vertex at the origin
    if (nd == 0.0) return;
    const double s = fast_div(f.ring_c, nd);
    if (!(s > 0.0) || !(s < INFINITY)) return;
    const V3 X = s * ov;
    const V3 tv = obsvec2targvec(fs, X);
    double lon, lat, alt;
    recpgr(fs, tv, false, lon, lat, alt);
    radius = alt + f.r_eq;
    lon_deg = lon * kDpr;
    dist = norm(X);
}

// Body._limb_coordinates_from_obsvec (body.py:2081-2110); ov finite
PM_HD void limb_coordinates(const FrameD &fs, V3 ov, double &lon_deg, double &lat_deg, double &dist) {
    const PMFrame &f = fs.f;
    lon_deg = lat_deg = dist = NAN;
    const double n2 = dot(ov, ov);
    if (!(n2 > 0.0)) return;
    const V3 u = fast_rsqrt(n2) * ov;  // spice.nplnpt(origin, ov, target centre)
    const V3 P0 = ld3(f.P0);
    const V3 pn = dot(P0, u) * u;
    const double near_dist = norm(P0 - pn);
    const V3 tv = obsvec2targvec(fs, pn);
    // spice.surfpt(origin, tv, a, b, c): radial surface point
    const V3 x = mul3(tv, fs.inv_r);
    const double xn2 = dot(x, x);
    if (!(xn2 > 0.0)) return;
    const V3 sp = fast_rsqrt(xn2) * tv;
    double lon, lat, alt;
    recpgr(fs, sp, fs.biaxial != 0, lon, lat, alt);
    lon_deg = lon * kDpr;
    lat_deg = lat * kDpr;
    dist = near_dist - norm(sp);
}

// ---------------------------------------------------------------------------------
// Plane ids / masks
// ---------------------------------------------------------------------------------
PM_HD constexpr uint64_t bit(int k) { return 1ull << k; }
constexpr uint64_t kKmMask = bit(PM_KM_X) | bit(PM_KM_Y) | bit(PM_ANGULAR_X) | bit(PM_ANGULAR_Y);
constexpr uint64_t kLonLatMask = bit(PM_LON_GRAPHIC) | bit(PM_LAT_GRAPHIC) | bit(PM_LOCAL_SOLAR_TIME);
constexpr uint64_t kCentricMask = bit(PM_LON_CENTRIC) | bit(PM_LAT_CENTRIC);
constexpr uint64_t kIllumMask = bit(PM_PHASE) | bit(PM_INCIDENCE) | bit(PM_EMISSION) | bit(PM_AZIMUTH);
constexpr uint64_t kStateMask = bit(PM_DISTANCE) | bit(PM_RADIAL_VELOCITY) | bit(PM_DOPPLER);
constexpr uint64_t kLimbMask = bit(PM_LIMB_DISTANCE) | bit(PM_LIMB_LON_GRAPHIC) | bit(PM_LIMB_LAT_GRAPHIC);
constexpr uint64_t kRingMask = bit(PM_RING_RADIUS) | bit(PM_RING_LON_GRAPHIC) | bit(PM_RING_DISTANCE);
constexpr uint64_t kSurfMask = kLonLatMask | kCentricMask | kIllumMask | kStateMask | kRingMask;
constexpr uint64_t kSkyMask = bit(PM_RA) | bit(PM_DEC) | kKmMask | kLimbMask | kRingMask;

// ---------------------------------------------------------------------------------
// Image direction: every requested backplane of one pixel.  `out.put(id, value)`
// receives each requested plane exactly once.
// Replaces the loops listed at pm_backplanes_img in include/pm_b200.h.
// ---------------------------------------------------------------------------------
// kSky = false compiles out RA / DEC / KM / ANGULAR / LIMB / RING planes (the launcher
// picks it when none is requested): smaller code, fewer registers for the default
// surface stack.
// kFixedMask != 0 fixes the plane set at compile time (the launcher uses it for the
// default surface stack): every `mask & bit` test folds away and the per-pixel code
// becomes a handful of large basic blocks the scheduler can interleave freely.
// kRingAll = true keeps ring-plane points hidden behind the body
// (Body.ring_plane_coordinates(only_visible=False), body.py:2577-2615); the backplanes hide them.
// kSpinSym = true is the path for frames with FrameD::spin_sym (the launchers pick it from the flag):
// the intercept, the illumination angles and the radial velocity are taken in the body frame at t_ref,
// where they equal the epoch frame's up to the bound of spin_sym, and only LON / LAT spin the point.
template <bool kSky, uint64_t kFixedMask = 0, bool kRingAll = false, bool kSpinSym = false, class Sink>
PM_HD void image_pixel(const FrameD &fs, double x, double y, uint64_t mask_in, Sink &out) {
    const PMFrame &f = fs.f;
    const double nan = NAN;
    const uint64_t mask = kFixedMask ? kFixedMask : (kSky ? mask_in : (mask_in & ~kSkyMask));
    if (mask & bit(PM_PIXEL_X)) out.put(PM_PIXEL_X, x);  // BodyXY.get_x_img / get_y_img (body_xy.py:3494-3531)
    if (mask & bit(PM_PIXEL_Y)) out.put(PM_PIXEL_Y, y);

    // BodyXY._get_targvec_img's early-out circle (body_xy.py:3201-3203): pixels outside it
    // never reach sincpt, and without sky planes they do not need the ray at all
    const double dx = x - f.x0, dy = y - f.y0;
    const bool try_disc = (mask & kSurfMask) && !(f.optimize_speed != 0.0 && fma(dx, dx, dy * dy) > f.r_cut2);
    V3 v = mk(nan, nan, nan);
    if (try_disc || (kSky && (mask & kSkyMask))) v = xy2ray_local(fs, x, y);
    V3 d2 = mk(nan, nan, nan);
    if (kSky && (mask & kSkyMask)) {
        // BodyXY._get_radec_img (body_xy.py:3413-3418)
        const V3 d = mtxv(f.M, v);
        double ra, dec;
        recrad_angles(d, ra, dec);
        const double ra_deg = ra * kDpr, dec_deg = dec * kDpr;
        if (mask & bit(PM_RA)) out.put(PM_RA, ra_deg);
        if (mask & bit(PM_DEC)) out.put(PM_DEC, dec_deg);
        // _get_obsvec_norm_img (body_xy.py:3263-3272): RA/Dec degrees -> unit vector
        if (mask & (kKmMask | kLimbMask | kRingMask)) d2 = radrec1(ra_deg * kRpd, dec_deg * kRpd);
        if (mask & kKmMask) {  // _get_km_xy_img (body_xy.py:3547-3553), angular (:3611-3656)
            double ax, ay;
            obsvec2angular(f, d2, ax, ay);
            const double kx = fma(f.ang2km[0], ax, f.ang2km[1] * ay);
            const double ky = fma(f.ang2km[2], ax, f.ang2km[3] * ay);
            if (mask & bit(PM_KM_X)) out.put(PM_KM_X, kx);
            if (mask & bit(PM_KM_Y)) out.put(PM_KM_Y, ky);
            if (mask & bit(PM_ANGULAR_X)) out.put(PM_ANGULAR_X, fast_div(kx, f.km_per_arcsec));
            if (mask & bit(PM_ANGULAR_Y)) out.put(PM_ANGULAR_Y, fast_div(ky, f.km_per_arcsec));
        }
    }

    // BodyXY._get_targvec_img (body_xy.py:3197-3225) incl. the early-out circle
    bool on_disc = false;
    Intercept it;
    const V3 u0 = mxv(fs.G, v);  // unit ray, body frame at t_ref
    if (try_disc) on_disc = sincpt<kSpinSym>(fs, u0, it);

    double v_dist = nan;
    if (on_disc) {
        const V3 p = it.p;
        if (mask & (kLonLatMask | kCentricMask)) {
            // _get_lonlat_img (body_xy.py:3284-3288), _get_lonlat_centric_img (:3349): the
            // east longitude and the cylindrical radius are shared by recpgr and reclat
            const double rho = fast_sqrt_lite(fma(p.x, p.x, p.y * p.y));
            const double lon_e = fast_atan2(p.y, p.x);
            if (mask & kLonLatMask) {
                double l = f.lon_sign * lon_e;
                if (l < 0.0) l += kTwoPi;
                const double v_lon = l * kDpr;
                double lat, alt;
                if (fs.biaxial) {
                    lat = fast_atan2_xpos(p.z * fs.inv_omf2, rho);
                } else {
                    geodetic_general(fs, rho, p.z, lat, alt);
                }
                if (mask & bit(PM_LON_GRAPHIC)) out.put(PM_LON_GRAPHIC, v_lon);
                if (mask & bit(PM_LAT_GRAPHIC)) out.put(PM_LAT_GRAPHIC, lat * kDpr);
                if (mask & bit(PM_LOCAL_SOLAR_TIME)) out.put(PM_LOCAL_SOLAR_TIME, local_solar_time(f, v_lon));
            }
            if (mask & bit(PM_LON_CENTRIC)) out.put(PM_LON_CENTRIC, lon_e * kDpr);
            if (mask & bit(PM_LAT_CENTRIC)) out.put(PM_LAT_CENTRIC, fast_atan2_xpos(p.z, rho) * kDpr);
        }
        if (mask & (kIllumMask | kStateMask | kRingMask)) {
            // spkcpt's converged light time is the intercept's own: |X| = |p - o|
            const V3 kxp = cross(ld3(fs.k), kSpinSym ? it.p0 : p);  // shared by the inverse spin and omega x p
            const V3 p0 = kSpinSym ? it.p0 : spin_bwd_c(fs, it.r, p, kxp);
            if (mask & kIllumMask) {  // _get_illumination_gie_img (body_xy.py:3661-3665)
                Illum il;
                if (kSpinSym)  // the angles of (n, s, e) all spun back to t_ref
                    illum_angles(mul3(p0, fs.nw), sun_vec0(fs, p0, it.dt), -u0, (mask & bit(PM_AZIMUTH)) != 0, il);
                else
                    illum_at(fs, p, p0, -it.u, it.r, it.dt, (mask & bit(PM_AZIMUTH)) != 0, il);
                if (mask & bit(PM_PHASE)) out.put(PM_PHASE, il.phase * kDpr);
                if (mask & bit(PM_INCIDENCE)) out.put(PM_INCIDENCE, il.incdnc * kDpr);
                if (mask & bit(PM_EMISSION)) out.put(PM_EMISSION, il.emissn * kDpr);
                if (mask & bit(PM_AZIMUTH)) out.put(PM_AZIMUTH, il.azimuth * kDpr);  // get_azimuth_angle_img (:3744)
            }
            v_dist = it.lt * f.clight;  // get_distance_img (body_xy.py:3870-3880)
            if (mask & bit(PM_DISTANCE)) out.put(PM_DISTANCE, v_dist);
            if (mask & (bit(PM_RADIAL_VELOCITY) | bit(PM_DOPPLER))) {
                // get_radial_velocity_img (body_xy.py:3898-3913): project on the line of sight - the pixel's
                // own ray (u0 in the frame of t_ref, it.u at the intercept epoch; the spin about k leaves
                // (k x p) . u unchanged, so the spin-symmetric path takes both at t_ref)
                const V3 vt = axpy(it.dt, ld3(fs.ATb), ld3(fs.VTb));
                const double a = fma(fs.wn, dot(kxp, kSpinSym ? u0 : it.u), dot(vt, u0));
                const double b = dot(ld3(fs.VOb), u0);
                const double rv = radial_velocity(fs, a, b);
                if (mask & bit(PM_RADIAL_VELOCITY)) out.put(PM_RADIAL_VELOCITY, rv);
                if (mask & bit(PM_DOPPLER)) out.put(PM_DOPPLER, doppler_factor(fs, rv));
            }
        }
    } else {
        const uint64_t m = mask & (kLonLatMask | kCentricMask | kIllumMask | kStateMask);
#pragma unroll
        for (int k = 0; k <= PM_DOPPLER; k++)
            if ((kLonLatMask | kCentricMask | kIllumMask | kStateMask) & bit(k))
                if (m & bit(k)) out.put(k, nan);
    }

    if (kSky && (mask & kLimbMask)) {  // _get_limb_coordinate_imgs (body_xy.py:3967-3975)
        double llon, llat, ldist;
        limb_coordinates(fs, d2, llon, llat, ldist);
        if (mask & bit(PM_LIMB_DISTANCE)) out.put(PM_LIMB_DISTANCE, ldist);
        if (mask & bit(PM_LIMB_LON_GRAPHIC)) out.put(PM_LIMB_LON_GRAPHIC, llon);
        if (mask & bit(PM_LIMB_LAT_GRAPHIC)) out.put(PM_LIMB_LAT_GRAPHIC, llat);
    }
    if (kSky && (mask & kRingMask)) {  // _get_ring_plane_coordinate_imgs (body_xy.py:4061-4085)
        double rad, rl, rd;
        ring_coordinates(fs, d2, rad, rl, rd);
        if (!kRingAll && rd > v_dist) rad = rl = rd = nan;  // NaN distance compares false (quirk kept)
        if (mask & bit(PM_RING_RADIUS)) out.put(PM_RING_RADIUS, rad);
        if (mask & bit(PM_RING_LON_GRAPHIC)) out.put(PM_RING_LON_GRAPHIC, rl);
        if (mask & bit(PM_RING_DISTANCE)) out.put(PM_RING_DISTANCE, rd);
    }
}

// The image-direction planes at one arbitrary image position (pm_backplanes_points_host): a
// fractional pixel, or one outside the image.  A non-finite x or y never reaches image_pixel -
// a NaN ray would drive sincpt's light-time iteration, which runs until the epoch stops
// changing - so it writes NaN to every plane, with PIXEL-X / PIXEL-Y echoing the input.
template <bool kSky, bool kRingAll, bool kSpinSym = false, class Sink>
PM_HD void image_point(const FrameD &fs, double x, double y, uint64_t mask_in, Sink &out) {
    if (fabs(x) < INFINITY && fabs(y) < INFINITY) {
        image_pixel<kSky, 0, kRingAll, kSpinSym>(fs, x, y, mask_in, out);
        return;
    }
#pragma unroll 1
    for (int k = 0; k < PM_N_PLANES; k++)
        if (mask_in & bit(k)) out.put(k, k == PM_PIXEL_X ? x : (k == PM_PIXEL_Y ? y : (double)NAN));
}

// ---------------------------------------------------------------------------------
// Map direction: the same quantities on one planetographic lon/lat cell, plus the
// inverse mapping cell -> image xy with the reference's visibility test.
// Replaces the loops listed at pm_backplanes_map in include/pm_b200.h.
// ---------------------------------------------------------------------------------
// kFixedMask != 0 fixes the plane set at compile time (the x / y map of map_img needs only the
// emission angle of illumf: phase, incidence and the state are then dead code).
template <uint64_t kFixedMask = 0, class Sink>
PM_HD void map_cell(const FrameD &fs, double lon_deg, double lat_deg, uint64_t mask_in, Sink &out) {
    const uint64_t mask = kFixedMask ? kFixedMask : mask_in;
    const PMFrame &f = fs.f;
    const double nan = NAN;
    // BodyXY._get_lonlat_map (body_xy.py:3293-3300)
    const double lonm = (fabs(lon_deg) < INFINITY) ? pymod360(lon_deg) : nan;
    const double latm = (fabs(lat_deg) < INFINITY) ? lat_deg : nan;
    if (mask & bit(PM_LON_GRAPHIC)) out.put(PM_LON_GRAPHIC, lonm);
    if (mask & bit(PM_LAT_GRAPHIC)) out.put(PM_LAT_GRAPHIC, latm);
    const bool lon_ok = lonm == lonm;
    const bool ok = lon_ok && (latm == latm);
    if (mask & bit(PM_LOCAL_SOLAR_TIME))  // get_local_solar_time_map (body_xy.py:3812)
        out.put(PM_LOCAL_SOLAR_TIME, lon_ok ? local_solar_time(f, lonm) : nan);

    double v_clon = nan, v_clat = nan, v_g = nan, v_i = nan, v_e = nan, v_az = nan, v_dist = nan, v_rv = nan,
           v_dop = nan, v_ra = nan, v_dec = nan, v_x = nan, v_y = nan, v_kx = nan, v_ky = nan, v_ax = nan,
           v_ay = nan;
    double limb_lon = nan, limb_lat = nan, limb_dist = nan, ring_rad = nan, ring_lon = nan, ring_dist = nan;
    if (ok) {
        const V3 tv = pgrrec0(fs, lonm * kRpd, latm * kRpd);  // _get_targvec_map (:3230)
        if (mask & kCentricMask) {                              // _get_lonlat_centric_map (:3357)
            double lo, la;
            reclat_angles(tv, lo, la);
            v_clon = lo * kDpr;
            v_clat = la * kDpr;
        }
        PointGeom g;
        point_geom(fs, tv, g);  // _get_illumf_map (:3671), _get_state_maps (:3851)
        Illum il;
        // point -> observer in the epoch frame = spin_fwd(-X0)
        illum_at(fs, tv, g.p0, spin_fwd(fs, g.r, -g.X0), g.r, g.dt, (mask & bit(PM_AZIMUTH)) != 0, il);
        v_g = il.phase * kDpr;
        v_i = il.incdnc * kDpr;
        v_e = il.emissn * kDpr;
        if (mask & bit(PM_AZIMUTH)) v_az = il.azimuth * kDpr;
        v_dist = g.lt * f.clight;
        if (mask & (bit(PM_RADIAL_VELOCITY) | bit(PM_DOPPLER))) {
            v_rv = point_rv(fs, tv, g);
            v_dop = doppler_factor(fs, v_rv);
        }
        const bool visibl = il.emissn < kHalfPi, lit = il.incdnc < kHalfPi;
        const uint64_t vis_mask = bit(PM_RA) | bit(PM_DEC) | bit(PM_PIXEL_X) | bit(PM_PIXEL_Y) | kKmMask;
        const bool want_vis = visibl && (mask & vis_mask), want_lit = lit && (mask & (kLimbMask | kRingMask));
        if (want_vis || want_lit) {
            const V3 ov = targvec2obsvec(fs, tv);  // _get_obsvec_map (:3275)
            if (want_vis) {
                double ra, dec;  // _get_radec_map (:3423-3432)
                recrad_angles(ov, ra, dec);
                v_ra = ra * kDpr;
                v_dec = dec * kDpr;
                if (mask & (vis_mask & ~(bit(PM_RA) | bit(PM_DEC)))) {
                    const V3 d2 = radrec1(v_ra * kRpd, v_dec * kRpd);
                    double ax, ay;
                    obsvec2angular(f, d2, ax, ay);
                    // _get_xy_map (:3482-3491) with _xy_in_image_frame (:1868)
                    const double x = fma(f.Ainv[0], ax, fma(f.Ainv[1], ay, f.Ainv[2]));
                    const double y = fma(f.Ainv[3], ax, fma(f.Ainv[4], ay, f.Ainv[5]));
                    if ((-0.5 < x && x < f.nx - 0.5) && (-0.5 < y && y < f.ny - 0.5)) {
                        v_x = x;
                        v_y = y;
                    }
                    v_kx = fma(f.ang2km[0], ax, f.ang2km[1] * ay);  // _get_km_xy_map (:3557)
                    v_ky = fma(f.ang2km[2], ax, f.ang2km[3] * ay);
                    if (mask & (bit(PM_ANGULAR_X) | bit(PM_ANGULAR_Y))) {
                        v_ax = fast_div(v_kx, f.km_per_arcsec);
                        v_ay = fast_div(v_ky, f.km_per_arcsec);
                    }
                }
            }
            // the reference tests `lit` (illumf[4]) here, not `visibl`
            // (body_xy.py:3981, :4097); reproduced as is
            if (lit && (mask & kLimbMask)) limb_coordinates(fs, ov, limb_lon, limb_lat, limb_dist);
            if (lit && (mask & kRingMask)) {
                ring_coordinates(fs, ov, ring_rad, ring_lon, ring_dist);
                if (ring_dist > v_dist) ring_rad = ring_lon = ring_dist = nan;
            }
        }
    }
    if (mask & bit(PM_LON_CENTRIC)) out.put(PM_LON_CENTRIC, v_clon);
    if (mask & bit(PM_LAT_CENTRIC)) out.put(PM_LAT_CENTRIC, v_clat);
    if (mask & bit(PM_RA)) out.put(PM_RA, v_ra);
    if (mask & bit(PM_DEC)) out.put(PM_DEC, v_dec);
    if (mask & bit(PM_PIXEL_X)) out.put(PM_PIXEL_X, v_x);
    if (mask & bit(PM_PIXEL_Y)) out.put(PM_PIXEL_Y, v_y);
    if (mask & bit(PM_KM_X)) out.put(PM_KM_X, v_kx);
    if (mask & bit(PM_KM_Y)) out.put(PM_KM_Y, v_ky);
    if (mask & bit(PM_ANGULAR_X)) out.put(PM_ANGULAR_X, v_ax);
    if (mask & bit(PM_ANGULAR_Y)) out.put(PM_ANGULAR_Y, v_ay);
    if (mask & bit(PM_PHASE)) out.put(PM_PHASE, v_g);
    if (mask & bit(PM_INCIDENCE)) out.put(PM_INCIDENCE, v_i);
    if (mask & bit(PM_EMISSION)) out.put(PM_EMISSION, v_e);
    if (mask & bit(PM_AZIMUTH)) out.put(PM_AZIMUTH, v_az);
    if (mask & bit(PM_DISTANCE)) out.put(PM_DISTANCE, v_dist);
    if (mask & bit(PM_RADIAL_VELOCITY)) out.put(PM_RADIAL_VELOCITY, v_rv);
    if (mask & bit(PM_DOPPLER)) out.put(PM_DOPPLER, v_dop);
    if (mask & bit(PM_LIMB_DISTANCE)) out.put(PM_LIMB_DISTANCE, limb_dist);
    if (mask & bit(PM_LIMB_LON_GRAPHIC)) out.put(PM_LIMB_LON_GRAPHIC, limb_lon);
    if (mask & bit(PM_LIMB_LAT_GRAPHIC)) out.put(PM_LIMB_LAT_GRAPHIC, limb_lat);
    if (mask & bit(PM_RING_RADIUS)) out.put(PM_RING_RADIUS, ring_rad);
    if (mask & bit(PM_RING_LON_GRAPHIC)) out.put(PM_RING_LON_GRAPHIC, ring_lon);
    if (mask & bit(PM_RING_DISTANCE)) out.put(PM_RING_DISTANCE, ring_dist);
}

// BodyXY._xy2lonlat (body_xy.py:482-496) -> Body._obsvec_norm2lonlat (body.py:1058-1081).
// Returns false when the ray misses the body (lon / lat left NaN).
PM_HD bool xy2lonlat_point(const FrameD &fs, double x, double y, double &lon, double &lat) {
    lon = lat = NAN;
    Intercept it;
    if (!sincpt(fs, mxv(fs.G, xy2ray_local(fs, x, y)), it)) return false;
    double lo, la, al;
    recpgr(fs, it.p, fs.biaxial != 0, lo, la, al);
    lon = lo * kDpr;
    lat = la * kDpr;
    return true;
}

// Body._lonlat2obsvec (body.py:1039-1056): planetographic (or planetocentric) lon / lat in degrees
// (+ altitude) -> the point as seen from the observer, J2000.  Returns false when the point is
// hidden (not_visible_nan).  Visibility: alt == 0 via illumf.visibl (body.py:2124-2130); alt != 0
// via the ray cast of Body._test_if_targvec_visible (body.py:2131-2150): hidden iff the ray
// observer -> point meets the surface and the surface is nearer.  planetocentric inputs go through
// spice.latsrf + recpgr first (Body._centric2graphic_lonlat, body.py:2966-2982).  lo / la receive
// the planetographic coordinates (radians) the point was built from, tv the body-fixed point.
PM_HD bool lonlat2obsvec_point(const FrameD &fs, double lon, double lat, double alt, bool not_visible_nan,
                               bool planetocentric, V3 &ov, double &lo, double &la, V3 &tv) {
    lo = lon * kRpd;
    la = lat * kRpd;
    if (planetocentric) {
        double sl, cl, sb, cb;
        sincos_full(lo, sl, cl);
        sincos_full(la, sb, cb);
        const V3 d = mk(cb * cl, cb * sl, sb);
        const V3 ds = mul3(d, fs.inv_r);
        const V3 sp = fast_rsqrt(dot(ds, ds)) * d;  // spice.latsrf on the ellipsoid
        double al;
        if (alt == 0.0) {
            recpgr(fs, sp, fs.biaxial != 0, lo, la, al);
        } else {
            // Body.targvec2lonlat(targvec, alt=alt) (body.py:1279-1283): recpgr against the
            // spheroid with every radius raised by alt (_AdjustedSurfaceAltitude, :210-229)
            lo = fs.f.lon_sign * fast_atan2(sp.y, sp.x);
            if (lo < 0.0) lo += kTwoPi;
            la = geodetic_lat_spheroid(fs.f.re + alt, fs.rp + alt, fast_sqrt(fma(sp.x, sp.x, sp.y * sp.y)), sp.z);
        }
        lo = (lo * kDpr) * kRpd;  // Body.targvec2lonlat returns degrees
        la = (la * kDpr) * kRpd;
    }
    tv = pgrrec0(fs, lo, la);
    if (alt != 0.0) {  // spice.pgrrec with an altitude: along the spheroid normal
        double sl, cl, sb, cb;
        sincos_full(fs.f.lon_sign * lo, sl, cl);
        sincos_full(la, sb, cb);
        tv = axpy(alt, mk(cb * cl, cb * sl, sb), tv);
    }
    if (not_visible_nan) {
        PointGeom g;
        point_geom(fs, tv, g);
        if (alt == 0.0) {
            // emission < pi/2  <=>  n . (point -> observer) > 0; evaluated as the angle itself
            // so that grazing cells agree with the map kernel
            const V3 e = spin_fwd(fs, g.r, -g.X0);
            const V3 n = mul3(tv, fs.nw);
            if (!(fast_atan2_ypos(norm(cross(n, e)), dot(n, e)) < kHalfPi)) return false;
        } else {
            Intercept it;
            const V3 dir = mxv(fs.f.R0, targvec2obsvec(fs, tv));
            if (sincpt(fs, fast_rsqrt(dot(dir, dir)) * dir, it)) {
                PointGeom gi;
                point_geom(fs, it.p, gi);
                if (!(g.lt < gi.lt)) return false;
            }
        }
    }
    ov = targvec2obsvec(fs, tv);
    return true;
}

// BodyXY._lonlat2xy (body_xy.py:544-560)
PM_HD void lonlat2xy_point(const FrameD &fs, double lon, double lat, double alt, bool not_visible_nan,
                           bool planetocentric, double &x, double &y) {
    x = y = NAN;
    V3 ov, tv;
    double lo, la;
    if (!lonlat2obsvec_point(fs, lon, lat, alt, not_visible_nan, planetocentric, ov, lo, la, tv)) return;
    if (!finite3(ov)) return;
    double ax, ay;
    obsvec2angular(fs.f, ov, ax, ay);
    x = fma(fs.f.Ainv[0], ax, fma(fs.f.Ainv[1], ay, fs.f.Ainv[2]));
    y = fma(fs.f.Ainv[3], ax, fma(fs.f.Ainv[4], ay, fs.f.Ainv[5]));
}

// ---------------------------------------------------------------------------------
// Generic point transform between the five coordinate systems of Body / BodyXY
// (SpiceBase._maybe_transform_as_arrays, base.py:718-757, around the scalar pairs
// Body.lonlat2radec ... Body.angular2km, body.py:1083-1900, and BodyXY.xy2radec ...
// angular2xy, body_xy.py:385-676).  Every pair goes through the observer-frame vector
// ("obsvec"), as in the reference.
// ---------------------------------------------------------------------------------
struct TransformAux {
    double Mc[9];      // obsvec -> angular rotation for the ANGULAR system (Body._get_obsvec2angular_matrix
                       // with the caller's origin_ra / origin_dec / coordinate_rotation; default = frame M)
    double km2ang[4];  // Body._get_km2angular_matrix (body.py:1625-1634)
};

// Body._obsvec2angular (body.py:1345-1361) with an explicit matrix, arcsec; ov finite
PM_HD void obsvec2angular_m(const double *M, V3 ov, double &ax, double &ay) {
    double ra, dec;
    recrad_angles(mxv(M, ov), ra, dec);
    double x = pymod360(-(ra * kDpr));
    if (x > 180.0) x -= 360.0;
    ax = x * 3600.0;
    ay = (dec * kDpr) * 3600.0;
}
// Body._angular2obsvec_norm (body.py:1363-1373)
PM_HD V3 angular2obsvec_m(const double *M, double ax, double ay) {
    return mtxv(M, radrec1(-((ax * (1.0 / 3600.0)) * kRpd), (ay * (1.0 / 3600.0)) * kRpd));
}

// Returns false only for a ray that misses the body on the way to lon / lat (counted by the caller).
PM_HD bool point_transform(const FrameD &fs, const TransformAux &aux, int src, int dst, double a, double b,
                           double alt, uint32_t flags, double &oa, double &ob) {
    const PMFrame &f = fs.f;
    oa = ob = NAN;
    if (!(fabs(a) < INFINITY) || !(fabs(b) < INFINITY)) return true;
    const bool pc = (flags & PM_FLAG_PLANETOCENTRIC) != 0;
    V3 ov;
    if (src == PM_COORD_LONLAT) {
        V3 tv;
        double lo, la;
        const bool vis = lonlat2obsvec_point(fs, a, b, alt, (flags & PM_FLAG_NOT_VISIBLE_NAN) != 0 &&
                                                              dst != PM_COORD_LONLAT && dst != PM_COORD_CENTRIC,
                                             pc, ov, lo, la, tv);
        if (dst == PM_COORD_LONLAT) {  // Body.centric2graphic_lonlat (body.py:2949-2982) / identity
            oa = lo * kDpr;
            ob = la * kDpr;
            return true;
        }
        if (dst == PM_COORD_CENTRIC) {  // Body.graphic2centric_lonlat (body.py:2915-2947): reclat of the point
            double lc, bc;
            reclat_angles(tv, lc, bc);
            oa = lc * kDpr;
            ob = bc * kDpr;
            return true;
        }
        if (!vis || !finite3(ov)) return true;
    } else if (src == PM_COORD_RADEC) {
        ov = radrec1(a * kRpd, b * kRpd);  // Body._radec2obsvec_norm (body.py:964-970)
    } else if (src == PM_COORD_ANGULAR) {
        ov = angular2obsvec_m(aux.Mc, a, b);
    } else if (src == PM_COORD_KM) {  // Body._km2obsvec_norm (body.py:1641-1644)
        ov = angular2obsvec_m(f.M, fma(aux.km2ang[0], a, aux.km2ang[1] * b), fma(aux.km2ang[2], a, aux.km2ang[3] * b));
    } else {  // BodyXY._xy2obsvec_norm (body_xy.py:375-377)
        ov = angular2obsvec_m(f.M, fma(f.A[0], a, fma(f.A[1], b, f.A[2])), fma(f.A[3], a, fma(f.A[4], b, f.A[5])));
    }
    if (!finite3(ov)) return true;
    if (dst == PM_COORD_RADEC) {  // SpiceBase._obsvec2radec (base.py:891-906)
        double ra, dec;
        recrad_angles(ov, ra, dec);
        oa = ra * kDpr;
        ob = dec * kDpr;
    } else if (dst == PM_COORD_ANGULAR) {
        obsvec2angular_m(aux.Mc, ov, oa, ob);
    } else if (dst == PM_COORD_KM) {  // Body._obsvec2km (body.py:1646-1650)
        double ax, ay;
        obsvec2angular_m(f.M, ov, ax, ay);
        oa = fma(f.ang2km[0], ax, f.ang2km[1] * ay);
        ob = fma(f.ang2km[2], ax, f.ang2km[3] * ay);
    } else if (dst == PM_COORD_XY) {  // BodyXY._obsvec2xy (body_xy.py:379-382)
        double ax, ay;
        obsvec2angular_m(f.M, ov, ax, ay);
        oa = fma(f.Ainv[0], ax, fma(f.Ainv[1], ay, f.Ainv[2]));
        ob = fma(f.Ainv[3], ax, fma(f.Ainv[4], ay, f.Ainv[5]));
    } else {  // Body._obsvec_norm2lonlat (body.py:1058-1081); the frame carries the radii raised by alt
        Intercept it;
        const V3 dir = mxv(f.R0, ov);
        if (!sincpt(fs, fast_rsqrt(dot(dir, dir)) * dir, it)) return false;
        double lo, la, al;
        recpgr(fs, it.p, fs.biaxial != 0, lo, la, al);
        oa = lo * kDpr;
        ob = la * kDpr;
        if (pc || dst == PM_COORD_CENTRIC) {
            // graphic2centric_lonlat(lon, lat, alt=alt) evaluated INSIDE the altitude adjustment
            // (body.py:1066-1080): pgrrec(lon, lat, alt) against the already raised spheroid, then reclat
            lo = oa * kRpd;
            la = ob * kRpd;
            V3 tv = pgrrec0(fs, lo, la);
            if (alt != 0.0) {
                double sl, cl, sb, cb;
                sincos_full(f.lon_sign * lo, sl, cl);
                sincos_full(la, sb, cb);
                tv = axpy(alt, mk(cb * cl, cb * sl, sb), tv);
            }
            double lc, bc;
            reclat_angles(tv, lc, bc);
            oa = lc * kDpr;
            ob = bc * kDpr;
        }
    }
    return true;
}

}  // namespace pm
