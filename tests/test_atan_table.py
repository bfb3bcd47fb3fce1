"""
The table-reduced arctangent of pm_math.cuh (atan_ratio: atan(t0) + atan(r) about t0 = k / 256, k from a
~20-bit reciprocal seed) on the inputs where a table reduction can go wrong: ratios at and beside every
rounding boundary (k + 1/2) / 256 of the index, the octant edge |y| = |x|, signed zeros and ratios down to
1e-300.  Every atan2 variant must stay within the 3-ulp bound of test_host_check / test_gpu_math, on the
host build (pessimistic truncated seeds) and on the device; the signed-zero conventions are exact.

Also FrameD::spin_z, the flag under which the spin-symmetric image path takes LON from the point at t_ref
less omega_z dt without spinning the point: on for Jupiter, Saturn and Venus, off beyond its 1e-8 km bound and
for a sphere whose spin axis is tilted off z, which keeps spin_sym and has to spin its points, so both paths
agree there as on the spheroids of test_spin_sym_host.py.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import img_case, triaxial_constants
from planetmapper_b200 import frame as F
from test_spin_sym_host import _bc, compare_paths, pixels, spin_lib, spin_sym  # noqa: F401 (fixture)

ATAN2, ATAN2_YPOS, ATAN2_XPOS = 5, 10, 11   # pm_math_probe kinds
SPINZ_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_check', 'host_check_spinz.cu')


def _edge_inputs():
    """(y, x) pairs: index boundaries, octant edges and extreme ratios, in all four quadrants and swapped"""
    k = np.arange(257, dtype=np.float64)
    rel = np.array([0.0, 2.0 ** -52, -2.0 ** -52, 2.0 ** -30, -2.0 ** -30, 2.0 ** -20, -2.0 ** -20, 2.0 ** -12,
                    -2.0 ** -12])
    q = np.concatenate([((k[:, None] + 0.5) / 256.0 * (1.0 + rel)).ravel(), (k[:, None] / 256.0 * (1.0 + rel)).ravel()])
    q = q[(q >= 0.0) & (q <= 1.0)]
    scale = np.array([1.0, 3.7e-5, 6.1e7, 1.0e-150, 1.0e150])
    x = np.repeat(scale, q.size)
    y = np.tile(q, scale.size) * x
    tiny = np.array([1e-300, 1e-200, 1e-100, 1e-20, 1e-9])
    y = np.concatenate([y, tiny, np.ones(tiny.size), tiny * 1e150])
    x = np.concatenate([x, np.ones(tiny.size), tiny, np.full(tiny.size, 1e150)])
    y, x = np.concatenate([y, x]), np.concatenate([x, y])   # the swapped octant
    sy = np.array([1.0, -1.0, 1.0, -1.0])
    sx = np.array([1.0, 1.0, -1.0, -1.0])
    return np.repeat(sy, y.size) * np.tile(y, 4), np.repeat(sx, x.size) * np.tile(x, 4)


def _max_ulp(got, want):
    want64 = want.astype(np.float64)
    ok = want64 != 0.0
    assert np.all(got[~ok] == 0.0)
    return float(np.max(np.abs(got[ok].astype(np.longdouble) - want[ok]) / np.spacing(np.abs(want64[ok]))))


def _check(run):
    y, x = _edge_inputs()
    yl, xl = y.astype(np.longdouble), x.astype(np.longdouble)
    report = {
        'atan2': _max_ulp(run(ATAN2, y, x), np.arctan2(yl, xl)),
        'atan2_ypos': _max_ulp(run(ATAN2_YPOS, y, x), np.arctan2(np.abs(yl), xl)),
        'atan2_xpos': _max_ulp(run(ATAN2_XPOS, y, x), np.arctan2(yl, np.abs(xl))),
    }
    print('edge-case ulp errors:', {k: round(v, 3) for k, v in report.items()})
    assert max(report.values()) <= 3.0, report
    # signed zeros and the axes, exactly
    zy = np.array([0.0, -0.0, 0.0, -0.0, 0.0, 1.0, -1.0, 2.5e-300, -7.0e200])
    zx = np.array([1.0, 1.0, -1.0, -1.0, 0.0, 0.0, -0.0, 0.0, -0.0])
    got = run(ATAN2, zy, zx)
    want = np.array([0.0, -0.0, np.pi, -np.pi, 0.0, np.pi / 2, -np.pi / 2, np.pi / 2, -np.pi / 2])
    assert np.array_equal(got, want) and np.array_equal(np.signbit(got), np.signbit(want)), got
    assert np.array_equal(run(ATAN2_YPOS, np.array([0.0, 0.0, 1.0]), np.array([1.0, -1.0, 0.0])),
                          np.array([0.0, np.pi, np.pi / 2]))
    assert np.array_equal(run(ATAN2_XPOS, np.array([1.0, -1.0, 0.0]), np.array([0.0, 0.0, 1.0])),
                          np.array([np.pi / 2, -np.pi / 2, 0.0]))
    assert np.isnan(run(ATAN2, np.array([np.nan, 1.0]), np.array([1.0, np.nan]))).all()


def test_atan2_edges_host(HC):
    def run(kind, y, x):
        y, x = np.ascontiguousarray(y), np.ascontiguousarray(x)
        out = np.empty_like(y)
        assert HC.hc_math(ctypes.c_int(kind), y.ctypes.data_as(ctypes.c_void_p), x.ctypes.data_as(ctypes.c_void_p),
                          ctypes.c_int64(y.size), out.ctypes.data_as(ctypes.c_void_p)) == 0
        return out

    _check(run)


@pytest.mark.gpu
def test_atan2_edges_device():
    import torch

    from planetmapper_b200 import _lib as L

    def run(kind, y, x):
        out = L.math_probe(kind, L.to_device(np.ascontiguousarray(y)), L.to_device(np.ascontiguousarray(x)))
        torch.cuda.synchronize()
        return out.cpu().numpy()

    _check(run)


@pytest.fixture(scope='module')
def spinz_lib(tmp_path_factory):
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not available')
    so = str(tmp_path_factory.mktemp('host_check_spinz') / 'libpm_hostcheck_spinz.so')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-shared', '-Xcompiler', '-fPIC', '-Wno-deprecated-gpu-targets',
                    '-o', so, SPINZ_SRC], check=True, capture_output=True)
    return ctypes.CDLL(so)


def spin_z(lib, fr):
    return bool(lib.hc_spin_z(np.ascontiguousarray(fr, dtype=np.float64).ctypes.data_as(ctypes.c_void_p)))


def _lon_shift_km(fr):
    """The displacement bound of FrameD::spin_z: |omega_perp| (2 a / clight) a"""
    w, r = F.frame_field(fr, 'omega'), F.frame_field(fr, 'radii')
    return float(np.hypot(w[0], w[1]) * 2.0 * r[0] / F.frame_field(fr, 'clight')[0] * r[0])


def test_spin_z_flag(spin_lib, spinz_lib, bc_hst):
    jup = img_case(bc_hst, 64, 48, 31.0, 24.5, 20.0, 17.0)
    assert spin_z(spinz_lib, jup) and 1e-9 < _lon_shift_km(jup) < 1e-8
    assert spin_z(spinz_lib, img_case(_bc('Saturn', 'EARTH'), 64, 48, 31.0, 24.5, 20.0, 17.0))
    assert spin_z(spinz_lib, img_case(_bc('Venus', 'EARTH'), 64, 48, 31.0, 24.5, 20.0, 17.0))
    for kind in ('europa', 'triaxial-x'):
        fr = img_case(triaxial_constants(kind), 64, 48, 31.0, 24.5, 20.0, 17.0)
        assert not spin_sym(spin_lib, fr) and not spin_z(spinz_lib, fr), kind
    # Jupiter with its spin axis tilted off z: spin_z follows the 1e-8 km bound, and never outlives spin_sym
    wn = float(np.linalg.norm(F.frame_field(jup, 'omega')))
    for tilt, want in ((1e-9, True), (3e-9, False), (1e-8, False)):   # 5.9e-9 km, 1.8e-8 km, 5.9e-8 km
        fr = jup.copy()
        F.frame_field(fr, 'omega')[:] = wn * np.array([np.sin(tilt), 0.0, np.cos(tilt)])
        assert (_lon_shift_km(fr) <= 1e-8) == want and spin_z(spinz_lib, fr) == want, tilt
        assert spin_sym(spin_lib, fr) or not want, tilt


def test_tilted_sphere_spins_its_points(spin_lib, spinz_lib):
    fr = img_case(_bc('Venus', 'EARTH'), 64, 48, 31.0, 24.5, 20.0, 17.0)
    w = F.frame_field(fr, 'omega')
    for tilt in (0.3, 2.0):
        w[:] = np.linalg.norm(w) * np.array([np.sin(tilt), 0.0, np.cos(tilt)])
        assert spin_sym(spin_lib, fr) and not spin_z(spinz_lib, fr), tilt
        print(compare_paths(spin_lib, fr, *pixels(64, 48, 31.0, 24.5, 20.0), f'venus tilted {tilt}'))
