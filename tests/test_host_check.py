"""
The kernels' own per-pixel / per-cell code (planetmapper_b200/csrc/pm_device.cuh is
__host__ __device__) instantiated on the CPU by tests/host_check/host_check.cu and
compared with the oracle with the SAME bars as the GPU parity tests.  This is the
no-GPU safety net for algorithmic changes to the device code; the GPU tests remain
the parity tests proper (the MUFU seeds are emulated here).  Test infrastructure only:
nothing in planetmapper_b200/ loads this library.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import (IMG_CASES, OTHER_BODIES, PID, TRIAXIAL_CASES, angle_diff, check_img_planes, check_map_planes,
                     assert_referee, close_observer_constants, img_case, random_geometry, triaxial_constants)
from planetmapper_b200 import frame as F

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'host_check', 'host_check.cu')
SO = os.path.join(HERE, 'host_check', '_build', 'libpm_hostcheck.so')
CSRC = os.path.join(os.path.dirname(HERE), 'planetmapper_b200', 'csrc')


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def hc_img(HC, fr, nx, ny, mask=(1 << 26) - 1):
    out = np.empty((26, ny, nx))
    f = np.ascontiguousarray(fr, dtype=np.float64)
    assert HC.hc_backplanes_img(_p(f), ctypes.c_int(nx), ctypes.c_int(ny), ctypes.c_uint64(mask), _p(out)) == 0
    return out


def hc_map(HC, fr, lon, lat, mask=(1 << 26) - 1):
    lon = np.ascontiguousarray(lon, dtype=np.float64)
    lat = np.ascontiguousarray(lat, dtype=np.float64)
    out = np.empty((26,) + lon.shape)
    f = np.ascontiguousarray(fr, dtype=np.float64)
    assert HC.hc_backplanes_map(_p(f), _p(lon), _p(lat), ctypes.c_int64(lon.size), ctypes.c_uint64(mask),
                                _p(out)) == 0
    return out


def _ulps(got, want):
    want = np.asarray(want, dtype=np.float64)
    return np.abs(got - want) / np.spacing(np.abs(want))


def test_math_primitives_ulp(HC):
    """pm_math.cuh on the host build (pessimistic 20-bit seeds) against numpy longdouble."""
    rng = np.random.default_rng(0)
    n = 400000
    a = (rng.uniform(-0.5, 0.5, n)) * 10.0 ** rng.uniform(-5, 15, n)
    b = (rng.uniform(-0.5, 0.5, n)) * 10.0 ** rng.uniform(-5, 15, n)
    al, bl = a.astype(np.longdouble), b.astype(np.longdouble)

    def run(kind, x, y=None):
        out = np.empty_like(x)
        assert HC.hc_math(ctypes.c_int(kind), _p(x), _p(y) if y is not None else None, ctypes.c_int64(x.size),
                          _p(out)) == 0
        return out

    def err(got, want):
        want = np.asarray(want)
        return float(np.max(np.abs(got.astype(np.longdouble) - want) / np.spacing(np.abs(want.astype(np.float64)))))

    assert err(run(0, a), 1 / al) <= 1.0
    assert err(run(7, a, b), al / bl) <= 1.0
    x = np.abs(a)
    assert err(run(1, x), 1 / np.sqrt(x.astype(np.longdouble))) <= 1.5
    assert err(run(2, x), np.sqrt(x.astype(np.longdouble))) <= 1.0
    th = rng.uniform(-np.pi / 4, np.pi / 4, n)
    assert err(run(3, th), np.sin(th.astype(np.longdouble))) <= 1.5
    assert err(run(4, th), np.cos(th.astype(np.longdouble))) <= 2.0
    assert err(run(5, a, b), np.arctan2(al, bl)) <= 3.0
    assert err(run(10, a, b), np.arctan2(np.abs(al), bl)) <= 3.0
    assert err(run(11, a, b), np.arctan2(al, np.abs(bl))) <= 3.0
    u = rng.uniform(-1, 1, n)
    u[::7] = 1 - 1e-9 * rng.uniform(0, 1, u[::7].size)
    assert err(run(6, u), np.arccos(u.astype(np.longdouble))) <= 4.0
    big = rng.uniform(-1000, 1000, n)
    assert np.max(np.abs(run(8, big) - np.sin(big.astype(np.longdouble)).astype(np.float64))) <= 3e-16
    assert np.max(np.abs(run(9, big) - np.cos(big.astype(np.longdouble)).astype(np.float64))) <= 3e-16
    # conventions the geometry relies on
    assert run(2, np.array([0.0]))[0] == 0.0
    assert run(5, np.array([0.0]), np.array([0.0]))[0] == 0.0
    assert run(5, np.array([0.0]), np.array([-1.0]))[0] == np.pi
    assert np.isnan(run(6, np.array([1.0000001]))[0]) and run(6, np.array([1.0]))[0] == 0.0


@pytest.mark.parametrize('case', sorted(IMG_CASES))
def test_device_code_image_planes_vs_oracle(HC, oracle, bc_hst, case):
    nx, ny, x0, y0, r0, rot, alt = IMG_CASES[case]
    fr = img_case(bc_hst, nx, ny, x0, y0, r0, rot, alt)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = hc_img(HC, fr, nx, ny)
    check_img_planes(got, ref, margin, fr, case)


def test_device_code_saturn_rings_vs_oracle(HC, oracle):
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), 'Saturn', '2004-12-30T12:00:00', 'EARTH')
    nx = ny = 96
    fr = img_case(bc, nx, ny, 47.5, 47.5, 18.0, 10.0)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = hc_img(HC, fr, nx, ny)
    check_img_planes(got, ref, margin, fr, 'saturn')


@pytest.mark.parametrize('target,observer,nx,ny,x0,y0,r0,rot', OTHER_BODIES)
def test_device_code_other_bodies_vs_oracle(HC, oracle, target, observer, nx, ny, x0, y0, r0, rot):
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), target, '2004-12-31T00:00:00', observer)
    fr = img_case(bc, nx, ny, x0, y0, r0, rot)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = hc_img(HC, fr, nx, ny)
    check_img_planes(got, ref, margin, fr, f'{target}/{observer}', allow_epoch_quantum=True)
    assert np.isfinite(got[PID['EMISSION']]).sum() > 0.3 * nx * ny * (r0 / max(nx, ny)) ** 2
    lons = np.arange(2.5, 360, 5.0)[::-1]
    lats = np.arange(-87.5, 90, 5.0)
    lo, la = np.meshgrid(lons, lats)
    refm, marginm = oracle.backplanes_map(fr, lo, la, with_margin=True)
    gotm = hc_map(HC, fr, lo, la)
    check_map_planes(gotm, refm, marginm, fr, nx, ny, f'{target}/{observer} map')


@pytest.mark.parametrize('nx,ny,x0,y0,r0,rot', [(10, 10, 5.0, 5.0, 3.0, 0.0), (120, 90, 61.0, 40.5, 55.0, 200.0)])
def test_device_code_close_observer_vs_oracle(HC, oracle, nx, ny, x0, y0, r0, rot):
    """Jupiter seen from Amalthea's distance (2.5 radii from the centre: the horizon is 67 deg from the
    sub-observer point, limb rays graze at large emission angles everywhere) - the geometry of the
    reference's test_mapping_visible_areas (tests/test_body_xy.py:2592-2608), on a synthetic orbit."""
    bc = close_observer_constants()
    assert 2.0 < bc.target_distance / max(bc.radii) < 3.0
    fr = img_case(bc, nx, ny, x0, y0, r0, rot)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = hc_img(HC, fr, nx, ny)
    check_img_planes(got, ref, margin, fr, 'jupiter/amalthea', allow_epoch_quantum=True)
    lo, la = np.meshgrid(np.arange(7.5, 360, 15.0)[::-1], np.arange(-82.5, 90, 15.0))
    refm, marginm = oracle.backplanes_map(fr, lo, la, with_margin=True)
    gotm = hc_map(HC, fr, lo, la)
    check_map_planes(gotm, refm, marginm, fr, nx, ny, 'jupiter/amalthea map')
    # visible part of the map <=> emission angle <= 90 deg <=> RA is defined (:2600-2605)
    emi, ra = gotm[PID['EMISSION']], gotm[PID['RA']]
    assert np.all(np.isfinite(ra[emi <= 90])) and not np.any(np.isfinite(ra[emi > 90]))
    assert 0.15 < np.isfinite(ra).mean() < 0.35     # a cap of 67 deg radius is 30 % of the sphere


@pytest.mark.parametrize('kind,nx,ny,x0,y0,r0,rot', TRIAXIAL_CASES)
def test_device_code_triaxial_vs_oracle(HC, oracle, kind, nx, ny, x0, y0, r0, rot):
    """Triaxial ellipsoids (Europa, and Europa's state with an exaggerated shape): image planes, map
    planes and the point transforms of the device code against the oracle."""
    bc = triaxial_constants(kind)
    fr = img_case(bc, nx, ny, x0, y0, r0, rot)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = hc_img(HC, fr, nx, ny)
    check_img_planes(got, ref, margin, fr, kind, allow_epoch_quantum=True)
    assert np.isfinite(got[PID['EMISSION']]).sum() > 500
    lo, la = np.meshgrid(np.arange(2.5, 360, 5.0)[::-1], np.arange(-87.5, 90, 5.0))
    refm, marginm = oracle.backplanes_map(fr, lo, la, with_margin=True)
    gotm = hc_map(HC, fr, lo, la)
    check_map_planes(gotm, refm, marginm, fr, nx, ny, f'{kind} map')
    f = np.ascontiguousarray(fr, dtype=np.float64)
    rng = np.random.default_rng(5)
    xs, ys = rng.uniform(0, nx - 1, 3000), rng.uniform(0, ny - 1, 3000)
    rl, rb, rmiss = oracle.xy2lonlat(fr, xs, ys)
    gl, gb = np.empty_like(xs), np.empty_like(xs)
    gmiss = ctypes.c_int64(0)
    assert HC.hc_xy2lonlat(_p(f), _p(xs), _p(ys), ctypes.c_int64(xs.size), _p(gl), _p(gb), ctypes.byref(gmiss)) == 0
    assert (np.isnan(gl) != np.isnan(rl)).sum() <= 2
    core = np.isfinite(gl) & np.isfinite(rl) & (np.hypot(xs - x0, ys - y0) < 0.7 * r0 * bc.radii[2] / bc.radii[0])
    assert core.sum() > 300
    # conditioning of a 1560 km body 8e8 km away: 2 ulp(|P0|) / r = 9e-9 deg per unit of 1 / cos(emission)
    # (helpers.surface_tolerances); the selected points have emission < 45 deg
    p0 = float(np.linalg.norm(F.frame_field(fr, 'P0')))
    bar = max(1e-9, 4.0 * np.rad2deg(2.0 * np.spacing(p0) / float(np.min(bc.radii))) * 1.5)
    assert np.max(np.abs(gb[core] - rb[core])) < bar
    assert np.max(angle_diff(gl[core], rl[core]) * np.cos(np.deg2rad(rb[core]))) < bar
    lon, lat = rng.uniform(0, 360, 3000), rng.uniform(-90, 90, 3000)
    for alt, pc in ((0.0, False), (12.5, False), (0.0, True), (-3.0, True)):
        rx, ry = oracle.lonlat2xy(fr, lon, lat, not_visible_nan=True, alt=alt, planetocentric=pc)
        gx, gy = np.empty_like(lon), np.empty_like(lon)
        assert HC.hc_lonlat2xy(_p(f), _p(lon), _p(lat), ctypes.c_int64(lon.size), ctypes.c_double(alt),
                               ctypes.c_uint32(1 | (4 if pc else 0)), _p(gx), _p(gy)) == 0
        assert (np.isnan(gx) != np.isnan(rx)).sum() <= 2, (alt, pc)
        ok = np.isfinite(rx) & np.isfinite(gx)
        assert ok.sum() > 500 or alt < 0   # points below the surface are always hidden
        if ok.any():
            assert np.max(np.abs(gx[ok] - rx[ok])) < 1e-9 * max(nx, ny)
            assert np.max(np.abs(gy[ok] - ry[ok])) < 1e-9 * max(nx, ny)


@pytest.mark.parametrize('target,observer', [('Moon', 'EARTH'), ('Venus', 'EARTH'), ('Jupiter', 'EARTH')])
def test_device_code_large_disc_limb_vs_oracle(HC, oracle, target, observer):
    """700-pixel discs: dozens of pixels with emission > 89.1 deg take sincpt's grazing-ray branch
    (light time iterated to convergence like CSPICE; the fixed three-pass scheme was off by up to 66
    tolerances on such pixels of the 2048 x 2048 frame)."""
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), target, '2004-12-31T00:00:00', observer)
    sz = 768
    fr = img_case(bc, sz, sz, 380.3, 390.7, 350.0, 33.0)
    ref, margin = oracle.backplanes_img(fr, sz, sz, with_margin=True)
    got = hc_img(HC, fr, sz, sz)
    check_img_planes(got, ref, margin, fr, f'{target}/{observer} 768', allow_epoch_quantum=True)
    assert (ref[PID['EMISSION']] > 89.1).sum() > 20


def test_device_code_plane_subsets(HC, bc_hst):
    fr = img_case(bc_hst, 60, 50, 29.5, 24.5, 22.0, 12.0)
    full = hc_img(HC, fr, 60, 50)
    for names in (['EMISSION'], ['LON-GRAPHIC', 'LAT-GRAPHIC'], ['RA', 'DEC', 'KM-X'], ['DOPPLER'],
                  ['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE', 'DISTANCE'],
                  ['LIMB-DISTANCE'], ['LOCAL-SOLAR-TIME'], ['AZIMUTH', 'PIXEL-X']):
        mask = sum(1 << PID[n] for n in names)
        sub = hc_img(HC, fr, 60, 50, mask)
        for n in names:
            assert np.array_equal(sub[PID[n]], full[PID[n]], equal_nan=True), n


@pytest.mark.parametrize('case', ['golden-7x10', 'rot-200x160', 'golden-7x10-alt'])
def test_device_code_map_planes_vs_oracle(HC, oracle, bc_hst, case):
    nx, ny, x0, y0, r0, rot, alt = IMG_CASES[case]
    fr = img_case(bc_hst, nx, ny, x0, y0, r0, rot, alt)
    lons = np.arange(1.5, 360, 3.0)[::-1]
    lats = np.arange(-88.5, 90, 3.0)
    lo, la = np.meshgrid(lons, lats)
    lo = lo.copy()
    lo[0, 0] = np.nan
    la[1, 1] = np.inf
    lo[2, 2] = -725.0
    ref, margin = oracle.backplanes_map(fr, lo, la, with_margin=True)
    got = hc_map(HC, fr, lo, la)
    check_map_planes(got, ref, margin, fr, nx, ny, case)


def test_device_code_point_transforms_vs_oracle(HC, oracle, bc_hst):
    fr = img_case(bc_hst, 15, 10, 5, 8, 3, 45)
    f = np.ascontiguousarray(fr, dtype=np.float64)
    rng = np.random.default_rng(1)
    xs = np.concatenate([rng.uniform(-2, 12, 4000), [np.nan, 5.0, np.inf, 5.0]])
    ys = np.concatenate([rng.uniform(2, 14, 4000), [8.0, np.nan, 8.0, 8.0]])
    rl, rb, rmiss = oracle.xy2lonlat(fr, xs, ys)
    gl, gb = np.empty_like(xs), np.empty_like(xs)
    gmiss = ctypes.c_int64(0)
    assert HC.hc_xy2lonlat(_p(f), _p(xs), _p(ys), ctypes.c_int64(xs.size), _p(gl), _p(gb), ctypes.byref(gmiss)) == 0
    assert (np.isnan(gl) != np.isnan(rl)).sum() <= 2 and abs(gmiss.value - rmiss) <= 2
    core = np.isfinite(gl) & np.isfinite(rl) & (np.hypot(xs - 5, ys - 8) < 2.5)
    assert np.max(np.abs(gb[core] - rb[core])) < 1e-9
    assert np.max(angle_diff(gl[core], rl[core]) * np.cos(np.deg2rad(rb[core]))) < 1e-9
    lon = np.concatenate([rng.uniform(-360, 720, 4000), [np.nan, 0.0, np.inf]])
    lat = np.concatenate([rng.uniform(-90, 90, 4000), [0.0, np.nan, 0.0]])
    for nvn in (True, False):
        rx, ry = oracle.lonlat2xy(fr, lon, lat, not_visible_nan=nvn)
        gx, gy = np.empty_like(lon), np.empty_like(lon)
        assert HC.hc_lonlat2xy(_p(f), _p(lon), _p(lat), ctypes.c_int64(lon.size), ctypes.c_double(0.0),
                               ctypes.c_uint32(1 if nvn else 0), _p(gx), _p(gy)) == 0
        assert np.array_equal(np.isnan(gx), np.isnan(rx))
        ok = np.isfinite(rx)
        assert np.max(np.abs(gx[ok] - rx[ok])) < 1e-9 and np.max(np.abs(gy[ok] - ry[ok])) < 1e-9
        # points above the surface (ray-cast visibility) and planetocentric inputs
        for alt, pc in ((1234.5, False), (-300.0, False), (50000.0, False), (0.0, True), (2345.6, True),
                        (-150.0, True)):
            rx, ry = oracle.lonlat2xy(fr, lon, lat, not_visible_nan=nvn, alt=alt, planetocentric=pc)
            flags = (1 if nvn else 0) | (4 if pc else 0)
            assert HC.hc_lonlat2xy(_p(f), _p(lon), _p(lat), ctypes.c_int64(lon.size), ctypes.c_double(alt),
                                   ctypes.c_uint32(flags), _p(gx), _p(gy)) == 0
            mism = np.isnan(gx) != np.isnan(rx)
            assert mism.sum() <= 2, (alt, pc, int(mism.sum()))      # only limb grazers may flip
            ok = np.isfinite(rx) & np.isfinite(gx)
            assert ok.sum() > 1000 or (alt < 0 and nvn)   # points below the surface are always hidden
            if not ok.any():
                continue
            assert np.max(np.abs(gx[ok] - rx[ok])) < 1e-9 and np.max(np.abs(gy[ok] - ry[ok])) < 1e-9, (alt, pc)


# ---------------------------------------------------------------------------------
# Extended-precision referee.  The oracle (oracle/pm_oracle.c) is re-compiled with every
# `double` turned into an 80-bit `long double` (sed + <tgmath.h>; the build lives under
# tests/host_check/_build/), which evaluates the SAME algorithm with 11 more mantissa
# bits and without the FP64 epoch quantisation.  Neither FP64 evaluation can be "more
# right" than its distance to that result, so this pins how much of a kernel-vs-oracle
# difference is FP64 noise of the algorithm itself, and checks that the kernels' own
# formulation (secant third pass, atan2-based angles, MUFU-seeded primitives) is no
# further from it than the CSPICE-shaped oracle is.
# ---------------------------------------------------------------------------------
LD_DRV = r"""
#include <stdio.h>
#include <stdlib.h>
#include <stdint.h>
#include "pm_b200_ld.h"
int pmo_backplanes_img(const PMFrame *f, int nx, int ny, uint64_t mask, long double *out, long double *margin);
int pmo_backplanes_map(const PMFrame *f, const long double *lon, const long double *lat, int64_t n, uint64_t mask,
                       long double *out, long double *margin);
int main(int argc, char **argv) {
    double fd[PM_FRAME_NDOUBLES];
    FILE *fp = fopen(argv[1], "rb");
    if (!fp || fread(fd, 8, PM_FRAME_NDOUBLES, fp) != PM_FRAME_NDOUBLES) return 1;
    fclose(fp);
    PMFrame f;
    long double *fl = (long double *)&f;
    for (int i = 0; i < PM_FRAME_NDOUBLES; i++) fl[i] = fd[i];
    int nx = atoi(argv[2]), ny = atoi(argv[3]);
    size_t n = (size_t)nx * ny;
    long double *out = malloc(sizeof(long double) * 26 * n), *m = malloc(sizeof(long double) * n);
    if (argc > 5) {   /* map direction: argv[5] holds n longitudes then n latitudes (doubles, degrees) */
        double *ll = malloc(16 * n);
        long double *lo = malloc(sizeof(long double) * n), *la = malloc(sizeof(long double) * n);
        fp = fopen(argv[5], "rb");
        if (!fp || fread(ll, 8, 2 * n, fp) != 2 * n) return 3;
        fclose(fp);
        for (size_t i = 0; i < n; i++) { lo[i] = ll[i]; la[i] = ll[n + i]; }
        if (pmo_backplanes_map(&f, lo, la, (int64_t)n, (1ull << 26) - 1, out, m)) return 2;
    } else if (pmo_backplanes_img(&f, nx, ny, (1ull << 26) - 1, out, m)) return 2;
    double *o = malloc(8 * 26 * n);
    for (size_t i = 0; i < 26 * n; i++) o[i] = (double)out[i];
    fp = fopen(argv[4], "wb");
    fwrite(o, 8, 26 * n, fp);
    fclose(fp);
    return 0;
}
"""


def write_ld_sources(bdir):
    """Writes the oracle with every `double` turned into an 80-bit `long double` into `bdir`: pm_oracle_ld.c and
    the headers it includes.  A driver declares what it calls from it (or includes the .c to reach its static
    routines) with "pm_b200_ld.h", whose PMFrame holds long doubles."""
    import re

    root = os.path.dirname(HERE)

    def ld(text):
        return re.sub(r'\bdouble\b', 'long double', text)
    c = ld(open(os.path.join(root, 'oracle', 'pm_oracle.c')).read()).replace('#include <math.h>', '#include <tgmath.h>')
    c = c.replace('#define PI 3.14159265358979323846264338327950288\n',
                  '#define PI 3.14159265358979323846264338327950288L\n')
    h = ld(open(os.path.join(root, 'oracle', 'pm_oracle.h')).read()).replace('"../include/pm_b200.h"', '"pm_b200_ld.h"')
    open(os.path.join(bdir, 'pm_oracle_ld.c'), 'w').write(c)
    open(os.path.join(bdir, 'pm_oracle.h'), 'w').write(h)
    open(os.path.join(bdir, 'pm_b200_ld.h'), 'w').write(ld(open(os.path.join(root, 'include', 'pm_b200.h')).read()))


def build_ld_oracle(bdir):
    """Compiles the oracle with every `double` turned into an 80-bit `long double` into `bdir` and
    returns run(frame, nx, ny) -> (26, ny, nx) planes (rounded to double at the very end)."""
    exe = os.path.join(bdir, 'oracle_ld')
    write_ld_sources(bdir)
    open(os.path.join(bdir, 'drv.c'), 'w').write(LD_DRV)
    subprocess.run(['gcc', '-O2', '-w', '-fopenmp', '-o', exe, 'drv.c', 'pm_oracle_ld.c', '-lm'], cwd=bdir, check=True,
                   capture_output=True)

    def run(fr, nx, ny, lonlat=None):
        """Image planes of an nx x ny frame, or (lonlat = (lon, lat) arrays) the map planes on those cells."""
        fin, fout = os.path.join(bdir, 'frame.bin'), os.path.join(bdir, 'out.bin')
        np.ascontiguousarray(fr, dtype=np.float64).tofile(fin)
        if lonlat is None:
            subprocess.run([exe, fin, str(nx), str(ny), fout], check=True)
            return np.fromfile(fout).reshape(26, ny, nx)
        lo, la = (np.ascontiguousarray(a, dtype=np.float64) for a in lonlat)
        fll = os.path.join(bdir, 'lonlat.bin')
        np.concatenate([lo.ravel(), la.ravel()]).tofile(fll)
        subprocess.run([exe, fin, str(lo.size), '1', fout, fll], check=True)
        return np.fromfile(fout).reshape((26,) + lo.shape)
    return run


@pytest.fixture(scope='module')
def ld_oracle(tmp_path_factory):
    if not shutil.which('gcc'):
        pytest.skip('gcc not available')
    return build_ld_oracle(str(tmp_path_factory.mktemp('oracle_ld')))   # always rebuilt from the current source


@pytest.mark.parametrize('target,observer,nx,ny,x0,y0,r0,rot', [('Jupiter', 'EARTH', 100, 100, 49.5, 49.5, 44.55, 0.0),
                                                               ('Venus', 'EARTH', 80, 64, 40.0, 30.0, 25.0, 15.0),
                                                               ('Moon', 'EARTH', 72, 72, 35.5, 35.5, 30.0, -20.0)])
def test_device_code_vs_extended_precision(HC, oracle, ld_oracle, target, observer, nx, ny, x0, y0, r0, rot):
    import planetmapper_b200 as pm
    from helpers import epoch_quantum_km

    bc = F.build_body_constants(pm.get_default_provider(), target, '2004-12-31T00:00:00', observer)
    fr = img_case(bc, nx, ny, x0, y0, r0, rot)
    exact = ld_oracle(fr, nx, ny)
    ref = oracle.backplanes_img(fr, nx, ny)
    got = hc_img(HC, fr, nx, ny)
    emi = exact[PID['EMISSION']]
    sel = np.isfinite(emi) & (emi < 70) & np.isfinite(got[PID['EMISSION']]) & np.isfinite(ref[PID['EMISSION']])
    assert sel.sum() > 500
    quantum = epoch_quantum_km(fr)
    r_min = float(np.min(F.frame_field(fr, 'radii')))
    report = {}
    for name in ('LON-GRAPHIC', 'LAT-GRAPHIC', 'EMISSION', 'INCIDENCE', 'PHASE', 'DISTANCE', 'RADIAL-VELOCITY'):
        k = PID[name]
        e_dev = np.abs(got[k][sel] - exact[k][sel])
        e_orc = np.abs(ref[k][sel] - exact[k][sel])
        report[name] = (float(e_dev.max()), float(e_orc.max()))
        # the kernels' formulation is no further from the extended-precision result than the oracle (up to a
        # thousandth of north_star's bar: below that both are rounding noise of the last FP64 operations)
        floor = 1e-15 if name in ('DISTANCE', 'RADIAL-VELOCITY') else 1e-12
        assert np.sqrt(np.mean(e_dev ** 2)) <= 1.5 * np.sqrt(np.mean(e_orc ** 2)) + floor, (name, report[name])
    # and both sit within ~one epoch quantum of relative motion of it (the FP64 noise floor of the path)
    assert report['DISTANCE'][0] <= 2.5 * quantum + 8 * np.spacing(float(np.linalg.norm(F.frame_field(fr, 'P0'))))
    ang_floor = np.rad2deg(2.5 * quantum / r_min) / np.cos(np.deg2rad(70.0)) ** 2 + 1e-10
    assert report['LAT-GRAPHIC'][0] <= ang_floor and report['EMISSION'][0] <= ang_floor
    print(target, {k: (f'{a:.2e}', f'{b:.2e}') for k, (a, b) in report.items()}, 'quantum km', quantum)


@pytest.mark.parametrize('block', range(6))
def test_device_code_random_geometries_vs_extended_precision(HC, oracle, ld_oracle, block):
    """Referee on random geometries far outside BASELINE.json's configs (observers from 1.3 to 1e5 radii,
    fields of view up to ~100 deg, six bodies): in every plane the kernels' per-pixel code is as close to
    the 80-bit evaluation of the reference algorithm as the FP64 oracle is.  This is the test that caught
    the secant error of the first intercept formulation for near observers."""
    for seed in range(16 * block, 16 * block + 16):
        fr, nx, ny, label = random_geometry(seed)
        ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
        assert_referee(hc_img(HC, fr, nx, ny), ref, ld_oracle(fr, nx, ny), margin, label)
        lo, la = np.meshgrid(np.arange(3.5, 360, 7.0)[::-1], np.arange(-87.5, 90, 5.0))
        refm, marginm = oracle.backplanes_map(fr, lo, la, with_margin=True)
        assert_referee(hc_map(HC, fr, lo, la), refm, ld_oracle(fr, nx, ny, (lo, la)), marginm, label + ' map',
                       xy_floor=1e-9 * max(nx, ny))   # 1e-9 of the frame, the bar of check_map_planes


def test_device_code_early_out_circle_flag(HC, oracle, bc_hst):
    """BodyXY(optimize_speed=...) (body_xy.py:3200-3217): pixels further than 1.05 r_max + 1 from the disc centre
    skip the intercept.  With the reference's radius the flag cannot change a result; with the cut-off radius
    shrunk INTO the disc (frame field r_cut2) the flag decides which pixels exist - the oracle and the kernel
    code must agree on both settings."""
    nx, ny = 64, 48
    frames = {}
    for opt in (True, False):
        fr = F.pack_frame(bc_hst, nx=nx, ny=ny, x0=30.0, y0=22.0, r0=18.0, rotation_radians=0.3, optimize_speed=opt)
        frames[opt] = fr
        ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
        check_img_planes(hc_img(HC, fr, nx, ny), ref, margin, fr, f'optimize_speed={opt}')
    a, b = hc_img(HC, frames[True], nx, ny), hc_img(HC, frames[False], nx, ny)
    assert np.array_equal(a, b, equal_nan=True)
    for opt in (True, False):
        fr = frames[opt].copy()
        F.frame_field(fr, 'r_cut2')[0] = 10.0 ** 2          # a view into the frame: cut the disc at 10 px
        ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
        got = hc_img(HC, fr, nx, ny)
        check_img_planes(got, ref, margin, fr, f'cut disc, optimize_speed={opt}')
        n_on = int(np.isfinite(got[PID['EMISSION']]).sum())
        assert (250 < n_on < 330) if opt else (n_on > 900), (opt, n_on)
