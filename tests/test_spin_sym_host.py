"""
The spin-symmetric path of the image-direction per-pixel code (image_pixel<..., kSpinSym = true>,
selected by FrameD::spin_sym) against the general path, both instantiated on the CPU by
tests/host_check/host_check_spin.cu.  For a spheroid spinning about its symmetry axis the two differ by
the neglected tilt of the spin axis (<= 1e-9 km by the flag's definition) and by rounding: the general
path spins the observer position (|P0| ~ 8e8 km for Jupiter), which moves it by about one ulp(|P0|).
So the NaN masks must be identical, and the planes agree to 1e-11 deg / 1e-13 relative plus ONE unit
of the positional noise of helpers.surface_tolerances (2 ulp(|P0|) + one epoch quantum, magnified by
1 / cos(emission)); the parity tests allow four units and a 1e-9 deg floor.  No GPU needed.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import (OTHER_BODIES, PID, angle_diff, close_observer_constants, epoch_quantum_km, img_case,
                     triaxial_constants)
from planetmapper_b200 import frame as F

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'host_check', 'host_check_spin.cu')
ALL = (1 << 26) - 1

ANGLES = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE', 'EMISSION', 'AZIMUTH']
ANGLE_BAR = 1e-11      # degrees
REL_BAR = 1e-13


@pytest.fixture(scope='module')
def spin_lib(tmp_path_factory):
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not available')
    so = str(tmp_path_factory.mktemp('host_check_spin') / 'libpm_hostcheck_spin.so')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-shared', '-Xcompiler', '-fPIC', '-Wno-deprecated-gpu-targets',
                    '-o', so, SRC], check=True, capture_output=True)
    return ctypes.CDLL(so)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def spin_sym(lib, fr):
    return bool(lib.hc_spin_sym(_p(np.ascontiguousarray(fr, dtype=np.float64))))


def run_path(lib, fr, x, y, sym):
    fr = np.ascontiguousarray(fr, dtype=np.float64)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    out = np.empty((26, x.size))
    assert lib.hc_backplanes_points_path(_p(fr), _p(x), _p(y), ctypes.c_int64(x.size), ctypes.c_uint64(ALL),
                                         ctypes.c_int(int(sym)), _p(out)) == 0
    return out


def pixels(nx, ny, x0, y0, r0, n_sample=None):
    """Every pixel, or (n_sample) a random sample plus every pixel of a 6-pixel annulus at the disc edge"""
    yy, xx = np.divmod(np.arange(nx * ny), nx)
    if n_sample is not None:
        keep = np.zeros(nx * ny, bool)
        keep[np.random.default_rng(0).choice(nx * ny, n_sample, replace=False)] = True
        keep |= np.abs(np.hypot(xx - x0, yy - y0) - r0) < 6.0
        xx, yy = xx[keep], yy[keep]
    return xx.astype(float), yy.astype(float)


def compare_paths(lib, fr, x, y, label):
    gen, sym = run_path(lib, fr, x, y, False), run_path(lib, fr, x, y, True)
    assert np.array_equal(np.isnan(gen), np.isnan(sym)), label
    on = np.isfinite(gen[PID['EMISSION']])
    assert on.sum() > 20, label
    # planes that do not read the intercept
    for name in ('RA', 'DEC', 'PIXEL-X', 'PIXEL-Y', 'KM-X', 'KM-Y', 'ANGULAR-X', 'ANGULAR-Y', 'LIMB-DISTANCE',
                 'LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC'):
        assert np.array_equal(gen[PID[name]], sym[PID[name]], equal_nan=True), (label, name)
    g = {n: gen[PID[n]][on] for n in PID}
    s = {n: sym[PID[n]][on] for n in PID}
    delta = 2.0 * np.spacing(float(np.linalg.norm(F.frame_field(fr, 'P0')))) + epoch_quantum_km(fr)   # km
    kappa = 1.0 / np.maximum(np.cos(np.deg2rad(g['EMISSION'])), 1e-12)
    ang = np.rad2deg(delta * kappa / float(np.min(F.frame_field(fr, 'radii'))))
    coslat = np.maximum(np.cos(np.deg2rad(g['LAT-CENTRIC'])), 1e-12)
    e, i = np.deg2rad(g['EMISSION']), np.deg2rad(g['INCIDENCE'])
    bars = {n: ANGLE_BAR + ang for n in ANGLES}
    bars['LON-GRAPHIC'] = bars['LON-CENTRIC'] = ANGLE_BAR + ang / coslat
    with np.errstate(divide='ignore'):   # the azimuth is undefined where e or i -> 0
        bars['AZIMUTH'] = ANGLE_BAR + ang * (1.0 / np.sin(e) + 1.0 / np.sin(i))
    bars['LOCAL-SOLAR-TIME'] = (ANGLE_BAR + ang / coslat) / 15.0   # hours
    bars['DISTANCE'] = REL_BAR * g['DISTANCE'] + delta * kappa
    wn = float(np.linalg.norm(F.frame_field(fr, 'omega')))
    bars['RADIAL-VELOCITY'] = REL_BAR * np.abs(g['RADIAL-VELOCITY']) + wn * delta * kappa + 1e-13
    bars['DOPPLER'] = bars['RADIAL-VELOCITY'] / 299792.458 + 4e-16
    report = {}
    for name, bar in bars.items():
        d = np.abs(g[name] - s[name])
        if name in ('LON-GRAPHIC', 'LON-CENTRIC'):
            d = angle_diff(g[name], s[name])
        elif name == 'LOCAL-SOLAR-TIME':
            d = np.minimum(d, 24.0 - d)
        report[name] = float(np.max(d / bar))
    assert max(report.values()) <= 1.0, (label, report)
    # ring planes: only their hiding test reads the intercept (its distance)
    for name in ('RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE'):
        ok = np.isfinite(gen[PID[name]])
        assert np.array_equal(gen[PID[name]][ok], sym[PID[name]][ok]), (label, name)
    return report


def _bc(target, observer, utc='2004-12-31T00:00:00'):
    import planetmapper_b200 as pm

    return F.build_body_constants(pm.get_default_provider(), target, utc, observer)


def test_paths_agree_on_the_c2_frame(spin_lib, bc_hst):
    sz = 2048
    c = (sz - 1) / 2
    fr = img_case(bc_hst, sz, sz, c, c, 0.9 * c, 0.0)
    assert spin_sym(spin_lib, fr)
    x, y = pixels(sz, sz, c, c, 0.9 * c, n_sample=30000)
    print(compare_paths(spin_lib, fr, x, y, 'C2'))


def test_paths_agree_on_saturn(spin_lib):
    fr = img_case(_bc('Saturn', 'EARTH', '2004-12-30T12:00:00'), 96, 96, 47.5, 47.5, 18.0, 10.0)
    assert spin_sym(spin_lib, fr)
    print(compare_paths(spin_lib, fr, *pixels(96, 96, 47.5, 47.5, 18.0), 'saturn'))


@pytest.mark.parametrize('target,observer,nx,ny,x0,y0,r0,rot', OTHER_BODIES)
def test_paths_agree_on_other_spheroids(spin_lib, target, observer, nx, ny, x0, y0, r0, rot):
    bc = _bc(target, observer)
    assert bc.radii[0] == bc.radii[1]
    fr = img_case(bc, nx, ny, x0, y0, r0, rot)
    assert spin_sym(spin_lib, fr)
    print(compare_paths(spin_lib, fr, *pixels(nx, ny, x0, y0, r0), f'{target}/{observer}'))


@pytest.mark.parametrize('nx,ny,x0,y0,r0,rot', [(10, 10, 5.0, 5.0, 3.0, 0.0), (120, 90, 61.0, 40.5, 55.0, 200.0)])
def test_paths_agree_for_a_close_observer(spin_lib, nx, ny, x0, y0, r0, rot):
    """Jupiter from 2.5 radii: limb rays graze everywhere and take sincpt's converging branch."""
    fr = img_case(close_observer_constants(), nx, ny, x0, y0, r0, rot)
    assert spin_sym(spin_lib, fr)
    print(compare_paths(spin_lib, fr, *pixels(nx, ny, x0, y0, r0), 'jupiter/amalthea'))


@pytest.mark.parametrize('target,observer', [('Moon', 'EARTH'), ('Venus', 'EARTH'), ('Jupiter', 'EARTH')])
def test_paths_agree_on_large_disc_limbs(spin_lib, target, observer):
    sz = 768
    fr = img_case(_bc(target, observer), sz, sz, 380.3, 390.7, 350.0, 33.0)
    assert spin_sym(spin_lib, fr)
    print(compare_paths(spin_lib, fr, *pixels(sz, sz, 380.3, 390.7, 350.0, n_sample=8000), f'{target}/{observer}'))


def _shift_km(fr):
    """The displacement bound of FrameD::spin_sym: |omega_perp| (2 a / clight) |a - c|"""
    w, r = F.frame_field(fr, 'omega'), F.frame_field(fr, 'radii')
    return float(np.hypot(w[0], w[1]) * 2.0 * r[0] / F.frame_field(fr, 'clight')[0] * abs(r[0] - r[2]))


def test_spin_sym_flag(spin_lib, bc_hst):
    jup = img_case(bc_hst, 64, 48, 31.0, 24.5, 20.0, 17.0)
    assert spin_sym(spin_lib, jup) and 0.0 < _shift_km(jup) < 1e-9
    assert spin_sym(spin_lib, img_case(_bc('Saturn', 'EARTH'), 64, 48, 31.0, 24.5, 20.0, 17.0))
    sphere = img_case(_bc('Venus', 'EARTH'), 64, 48, 31.0, 24.5, 20.0, 17.0)
    r = F.frame_field(sphere, 'radii')
    assert r[0] == r[1] == r[2] and spin_sym(spin_lib, sphere)
    # a sphere stays on whatever the tilt of its spin axis: nothing is neglected
    w = F.frame_field(sphere, 'omega')
    w[:] = np.linalg.norm(w) * np.array([np.sin(0.3), 0.0, np.cos(0.3)])
    assert spin_sym(spin_lib, sphere)
    for kind in ('europa', 'triaxial-x'):
        assert not spin_sym(spin_lib, img_case(triaxial_constants(kind), 64, 48, 31.0, 24.5, 20.0, 17.0)), kind
    # Jupiter with its spin axis tilted off the symmetry axis: on below the 1e-9 km bound, off above it
    wn = float(np.linalg.norm(F.frame_field(jup, 'omega')))
    for tilt, want in ((1e-9, True), (1e-8, False), (1e-3, False)):   # 3.9e-10 km, 3.9e-9 km, 0.4 m
        fr = jup.copy()
        F.frame_field(fr, 'omega')[:] = wn * np.array([np.sin(tilt), 0.0, np.cos(tilt)])
        assert (_shift_km(fr) <= 1e-9) == want and spin_sym(spin_lib, fr) == want, tilt


@pytest.mark.parametrize('target,observer,nx,ny,x0,y0,r0,rot', [('Jupiter', 'EARTH', 100, 100, 49.5, 49.5, 44.55, 0.0),
                                                               ('Venus', 'EARTH', 80, 64, 40.0, 30.0, 25.0, 15.0),
                                                               ('Earth', 'MOON', 64, 80, 30.0, 41.0, 26.0, 200.0)])
def test_spin_sym_path_vs_extended_precision(spin_lib, tmp_path, target, observer, nx, ny, x0, y0, r0, rot):
    """Neither path is the reference: against the 80-bit evaluation of the oracle's algorithm
    (test_host_check.build_ld_oracle) the spin-symmetric path is as close as the general one."""
    if not shutil.which('gcc'):
        pytest.skip('gcc not available')
    from test_host_check import build_ld_oracle

    fr = img_case(_bc(target, observer), nx, ny, x0, y0, r0, rot)
    exact = build_ld_oracle(str(tmp_path))(fr, nx, ny).reshape(26, -1)
    x, y = pixels(nx, ny, x0, y0, r0)
    gen, sym = run_path(spin_lib, fr, x, y, False), run_path(spin_lib, fr, x, y, True)
    sel = np.isfinite(exact[PID['EMISSION']]) & np.isfinite(gen[PID['EMISSION']])
    assert sel.sum() > 500
    for name in ('LON-GRAPHIC', 'LAT-GRAPHIC', 'EMISSION', 'INCIDENCE', 'PHASE', 'AZIMUTH', 'DISTANCE',
                 'RADIAL-VELOCITY'):
        k = PID[name]
        rms = [float(np.sqrt(np.mean(angle_diff(p[k][sel], exact[k][sel]) ** 2))) for p in (gen, sym)]
        assert rms[1] <= 1.1 * rms[0] + 1e-15, (name, rms)
