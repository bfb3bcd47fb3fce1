"""
CPU checks of the per-point geometry queries (Body.illumination_angles_from_lonlat ...
ring_plane_coordinates) and of pm_backplanes_points_host, the kernel behind the RA / Dec ones:
argument validation of the C entry point, the methods' host-side rules (alt refused before any
device work, the 'HH:MM:SS' form of the local solar time) and the host instantiation of the
per-point device code (tests/host_check/host_check_points.cu).  No GPU needed.
"""
import ctypes
import math
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from helpers import IMG_CASES, PID, img_case
from planetmapper_b200 import _lib as L
from planetmapper_b200 import body_xy as BX
from planetmapper_b200 import frame as F
from test_oracle_golden import RADEC_POINT_LITERALS, frame_looking_at

POINTS_SRC = os.path.join(ROOT, 'tests', 'host_check', 'host_check_points.cu')
ORACLE_POINTS_SRC = os.path.join(ROOT, 'tests', 'oracle_ext', 'oracle_points.c')


# ---- references for the point queries: the CPU oracle's routines driven point by point ------------------
class OraclePoints:
    """ctypes front of tests/oracle_ext/oracle_points.c (the unchanged oracle source plus two loops), built once
    per process into a temporary directory with the oracle's compiler flags."""

    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            import tempfile

            cc = '/usr/bin/gcc' if os.access('/usr/bin/gcc', os.X_OK) else (shutil.which('gcc') or 'gcc')
            so = os.path.join(tempfile.mkdtemp(prefix='oracle_points_'), 'liboracle_points.so')
            subprocess.run([cc, '-O2', '-fPIC', '-ffp-contract=off', '-std=c11', '-shared', '-o', so,
                            ORACLE_POINTS_SRC, '-lm'], check=True, capture_output=True)
            cls._lib = ctypes.CDLL(so)
        return cls._lib

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    @classmethod
    def backplanes_points(cls, frame, x, y, mask=L.ALL_PLANES, with_margin=False):
        """The oracle's image-direction planes at arbitrary finite positions (x, y): (popcount(mask),) + x.shape."""
        f = np.ascontiguousarray(frame, dtype=np.float64)
        x, y = (np.ascontiguousarray(a) for a in np.broadcast_arrays(np.asarray(x, dtype=np.float64),
                                                                     np.asarray(y, dtype=np.float64)))
        out, margin = np.empty((L.popcount(mask),) + x.shape), np.empty(x.shape)
        p = cls._p
        assert cls.lib().pmox_backplanes_points(p(f), p(x), p(y), ctypes.c_int64(x.size), ctypes.c_uint64(mask),
                                                p(out), p(margin)) == 0
        return (out, margin) if with_margin else out

    @classmethod
    def ring_coordinates(cls, frame, ra, dec):
        """Body.ring_plane_coordinates(ra, dec, only_visible=False) per direction: (radius, longitude, distance)."""
        f = np.ascontiguousarray(frame, dtype=np.float64)
        ra, dec = (np.ascontiguousarray(a) for a in np.broadcast_arrays(np.asarray(ra, dtype=np.float64),
                                                                        np.asarray(dec, dtype=np.float64)))
        radius, lon, dist = np.empty(ra.shape), np.empty(ra.shape), np.empty(ra.shape)
        p = cls._p
        assert cls.lib().pmox_ring_coordinates(p(f), p(ra), p(dec), ctypes.c_int64(ra.size), p(radius), p(lon),
                                               p(dist)) == 0
        return radius, lon, dist


# ---- pm_backplanes_points_host argument validation (no device work) ----------------------------------
def _frame_buf(bc):
    fr = np.ascontiguousarray(img_case(bc, 64, 48, 50.0, 10.0, 40.0, 200.0))
    return fr, fr.ctypes.data_as(ctypes.c_void_p)


def test_points_entry_validates_arguments_before_device_work(bc_hst):
    lib = L.load_library()
    fr, pf = _frame_buf(bc_hst)
    buf = np.zeros(8)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    f = lib.pm_backplanes_points_host
    assert f(pf, None, None, 0, L.ALL_PLANES, 0, None, None) == 0
    assert f(pf, None, None, 0, L.ALL_PLANES, L.FLAG_RING_ALL, None, None) == 0
    assert f(pf, None, None, 1, L.ALL_PLANES, 0, None, None) == -1
    assert f(pf, p, None, 1, L.ALL_PLANES, 0, p, None) == -1
    assert f(pf, None, p, 1, L.ALL_PLANES, 0, p, None) == -1
    assert f(pf, p, p, 1, L.ALL_PLANES, 0, None, None) == -1
    assert f(None, p, p, 1, L.ALL_PLANES, 0, p, None) == -1
    assert f(pf, p, p, -1, L.ALL_PLANES, 0, p, None) == -1
    assert f(pf, p, p, 1, 0, 0, p, None) == -1                   # no plane requested
    for bad in (1, 2, 4, 16, 1 << 31):                          # only PM_FLAG_RING_ALL is a flag here
        assert f(pf, p, p, 1, L.ALL_PLANES, bad, p, None) == -1, bad
        assert f(pf, None, None, 0, L.ALL_PLANES, bad, None, None) == -1, bad


# ---- host-side rules of the public methods ---------------------------------------------------------
LONLAT_METHODS = ['illumination_angles_from_lonlat', 'azimuth_angle_from_lonlat', 'distance_from_lonlat',
                  'radial_velocity_from_lonlat']


@pytest.fixture
def no_device(monkeypatch):
    """Any device work through the library wrappers fails the test."""
    def boom(*a, **k):
        raise AssertionError('device work before the argument checks')

    for name in ('to_device', 'backplanes_map_host', 'backplanes_points_host', 'transform', '_torch'):
        monkeypatch.setattr(L, name, boom)


@pytest.mark.parametrize('method', LONLAT_METHODS)
def test_nonzero_alt_is_refused_before_device_work(bc_hst, no_device, method):
    body = BX.BodyXY(constants=bc_hst)
    fn = getattr(body, method)
    with pytest.raises(NotImplementedError):
        fn(10.0, 20.0, alt=1.0)
    with pytest.raises(NotImplementedError):
        fn(np.zeros(5), np.zeros(5), alt=-3.0)


LST_LITERALS = [(22.89638888888889, '22:53:47'), (14.666111111111112, '14:39:58'), (4.896388888888889, '04:53:47'),
                (4.229722222222223, '04:13:47')]


def test_local_solar_time_string_of_the_literals():
    for hours, text in LST_LITERALS:
        assert BX.BodyXY._lst_string(hours) == text


@pytest.mark.parametrize('h,m,s', [(13, 0, 0), (12, 59, 0), (0, 0, 0), (23, 59, 59), (9, 30, 0), (1, 0, 59)])
def test_local_solar_time_string_near_boundaries(h, m, s):
    exact = h + m / 60 + s / 3600
    for eps in (-1e-9, -1e-12, 0.0, 1e-12, 1e-9):
        t = exact + eps
        if t < 0:
            continue
        assert BX.BodyXY._lst_string(t) == '%02d:%02d:%02d' % (h, m, s), (t, eps)


def test_local_solar_time_string_array_form(bc_hst, monkeypatch):
    body = BX.BodyXY(constants=bc_hst)
    hours = np.array([[v for v, _ in LST_LITERALS], [13 - 1e-9, 12 + 59 / 60 + 1e-9, 0.0, np.nan]])
    monkeypatch.setattr(body, 'local_solar_time_from_lon', lambda lon: hours)
    got = body.local_solar_time_string_from_lon(np.zeros((2, 4)))
    assert got.dtype == np.dtype('<U8') and got.shape == (2, 4)
    assert got[0].tolist() == [t for _, t in LST_LITERALS]
    assert got[1].tolist() == ['13:00:00', '12:59:00', '00:00:00', 'nan']
    monkeypatch.setattr(body, 'local_solar_time_from_lon', lambda lon: 22.89638888888889)
    assert body.local_solar_time_string_from_lon(0.0) == '22:53:47'


# ---- host instantiation of the per-point device code --------------------------------------------------
@pytest.fixture(scope='module')
def points_so(tmp_path_factory):
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not available')
    so = str(tmp_path_factory.mktemp('host_check_points') / 'libpm_hostcheck_points.so')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-shared', '-Xcompiler', '-fPIC', '-Wno-deprecated-gpu-targets',
                    '-o', so, POINTS_SRC], check=True, capture_output=True)
    return so


def _host_points(lib, fr, x, y, mask=L.ALL_PLANES, flags=0):
    fr = np.ascontiguousarray(fr, dtype=np.float64)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    out = np.empty((L.N_PLANES, x.size))
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    assert lib.hc_backplanes_points(p(fr), p(x), p(y), ctypes.c_int64(x.size), ctypes.c_uint64(mask),
                                    ctypes.c_uint32(flags), p(out)) == 0
    return out


_NONFINITE_SCRIPT = r'''
import ctypes, sys
import numpy as np
so, frame_path = sys.argv[1], sys.argv[2]
lib = ctypes.CDLL(so)
fr = np.load(frame_path)
nan, inf = np.nan, np.inf
x = np.array([nan, 31.0, inf, -inf, 31.0, 31.0, nan, 1e300])
y = np.array([24.5, nan, 24.5, 24.5, inf, -inf, nan, 24.5])
p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
no_sky = 0xFFFFF & ~0xF30   # planes 0-19 without RA / DEC / KM / ANGULAR: the kSky = false instantiation
for mask, flags in (((1 << 26) - 1, 0), ((1 << 26) - 1, 8), (no_sky, 0)):
    out = np.empty((26, x.size))
    assert lib.hc_backplanes_points(p(fr), p(x), p(y), ctypes.c_int64(x.size), ctypes.c_uint64(mask),
                                    ctypes.c_uint32(flags), p(out)) == 0
    for k in range(26):
        if k in (6, 7):   # PIXEL-X / PIXEL-Y echo the input
            assert np.array_equal(out[k][:7], (x if k == 6 else y)[:7], equal_nan=True), k
        else:
            assert np.isnan(out[k][:7]).all(), k
print('ok')
'''


def test_nonfinite_points_never_reach_the_intercept(bc_hst, points_so, tmp_path):
    """x or y NaN / +-inf: every plane NaN, PIXEL-X / PIXEL-Y echo the input, and the call returns.  Run in a
    child process with a time limit, so that a regression (a NaN ray in sincpt's light-time loop) fails the
    test instead of hanging the suite."""
    frame_path = str(tmp_path / 'frame.npy')
    np.save(frame_path, img_case(bc_hst, 64, 48, 31.0, 24.5, 20.0, 17.0))
    proc = subprocess.run([sys.executable, '-c', _NONFINITE_SCRIPT, points_so, frame_path], capture_output=True,
                          text=True, timeout=120)
    assert proc.returncode == 0 and proc.stdout.strip() == 'ok', proc.stderr[-2000:]


def test_host_points_equal_host_image_pixels(bc_hst, points_so, HC):
    """At integer positions, in shuffled order, the per-point code is the per-pixel code (host builds)."""
    lib = ctypes.CDLL(points_so)
    nx, ny, *rest = IMG_CASES['offset-disc-partly-outside']
    fr = img_case(bc_hst, nx, ny, *rest)
    want = np.empty((L.N_PLANES, ny * nx))
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    assert HC.hc_backplanes_img(p(fr), nx, ny, ctypes.c_uint64(L.ALL_PLANES), p(want)) == 0
    order = np.random.default_rng(1).permutation(nx * ny)
    got = _host_points(lib, fr, (order % nx).astype(float), (order // nx).astype(float))
    assert np.array_equal(got.view(np.int64), want[:, order].view(np.int64))


def test_host_ring_all_keeps_the_hidden_ring_point(bc_hst, points_so, oracle):
    """The ring point behind the disc (reference literal: NaN with only_visible=True) is kept by
    PM_FLAG_RING_ALL, lies beyond the body along the ray, and matches the oracle's unhidden coordinates."""
    lib = ctypes.CDLL(points_so)
    hidden = [rd for rd, exp in RADEC_POINT_LITERALS if all(v != v for v in exp.values()) and len(exp) == 3]
    assert hidden
    mask = L.mask_from_names(['DISTANCE', 'RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE'])
    for ra, dec in hidden:
        fr = frame_looking_at(bc_hst, ra, dec)
        vis = _host_points(lib, fr, [0.0], [0.0], mask)[:, 0]
        assert math.isnan(vis[PID['RING-RADIUS']]) and math.isfinite(vis[PID['DISTANCE']])
        allp = _host_points(lib, fr, [0.0], [0.0], mask, L.FLAG_RING_ALL)[:, 0]
        assert np.isfinite(allp[[PID['RING-RADIUS'], PID['RING-LON-GRAPHIC'], PID['RING-DISTANCE']]]).all()
        assert allp[PID['RING-DISTANCE']] > allp[PID['DISTANCE']]
        pra, pdec, _ = oracle.transform(fr, 'xy', 'radec', 0.0, 0.0)
        rad, lon, dist = (float(v[0]) for v in OraclePoints.ring_coordinates(fr, pra, pdec))
        p0 = float(np.linalg.norm(F.frame_field(fr, 'P0')))
        assert abs(allp[PID['RING-RADIUS']] - rad) <= 50e-12 * p0
        assert abs(allp[PID['RING-DISTANCE']] - dist) <= 50e-12 * p0
        # this ring point lies within a km of the body's centre: the bar of helpers.check_img_planes, which
        # scales with 1 / RING-RADIUS, applies to its longitude
        stretch = dist / float(F.frame_field(fr, 'ring_c')[0])
        d = abs(allp[PID['RING-LON-GRAPHIC']] - lon)
        assert min(d, 360 - d) <= max(1e-9, math.degrees(8 * np.spacing(p0) * stretch / max(abs(rad), 1.0)))


def test_oracle_points_entry_equals_its_image_entry_at_pixels(oracle, bc_hst):
    """OraclePoints.backplanes_points (the sub-pixel reference of the GPU tests) at integer positions is the
    oracle's image path, bit for bit."""
    nx, ny, *rest = IMG_CASES['golden-7x10-alt']
    fr = img_case(bc_hst, nx, ny, *rest)
    want, wmargin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    yy, xx = np.mgrid[0:ny, 0:nx].astype(float)
    got, margin = OraclePoints.backplanes_points(fr, xx, yy, with_margin=True)
    assert np.array_equal(got, want, equal_nan=True) and np.array_equal(margin, wmargin, equal_nan=True)
