"""
CPU checks of map_img's smoothing splines (spline_smoothing > 0): the host build of the fit that
pm_regrid_fit runs per plane (planetmapper_b200/csrc/pm_regrid.cuh, instantiated by
tests/host_check/host_check_regrid.cu) against scipy's FITPACK regrid, called with exactly the
arguments RectBivariateSpline(arange(ny), arange(nx), z, kx, ky, s) passes; the argument checks of the
new C entry points; and the host-side rules of map_img (degree refusal, scipy's ValueError text).
No GPU needed.

One class of inputs is left out of the exact comparison, counted and bounded: fits in which one axis
reaches its interpolation knot count (nx = mx + kx + 1 or ny = my + ky + 1) while the other is still
growing.  There the installed scipy's regrid overwrites a knot of the other axis that it never fitted
(a capped nyest probe of the same input aborts the interpreter with "double free or corruption"), so
its knots there are not FITPACK's algorithm but an out-of-bounds write.  Every other case must agree.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from planetmapper_b200 import _lib as L
from planetmapper_b200 import body_xy as BX

REGRID_SRC = os.path.join(ROOT, 'tests', 'host_check', 'host_check_regrid.cu')
SHAPES = [(7, 10), (16, 16), (64, 64), (128, 96), (33, 200)]
DEGREES = [(kx, ky) for kx in (1, 2, 3) for ky in (1, 2, 3)]


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope='module')
def regrid_so(tmp_path_factory):
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not available')
    so = str(tmp_path_factory.mktemp('host_check_regrid') / 'libpm_hostcheck_regrid.so')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-shared', '-Xcompiler', '-fPIC', '-Wno-deprecated-gpu-targets',
                    '-o', so, REGRID_SRC], check=True, capture_output=True)
    return ctypes.CDLL(so)


def host_fit(lib, z, kx, ky, s, nxest=None, nyest=None, maxit=20):
    """The host build of the device fit: (nx, tx, ny, ty, c, fp, ier) like scipy's regrid."""
    mx, my = z.shape
    nxest = nxest or mx + kx + 1
    nyest = nyest or my + ky + 1
    z = np.ascontiguousarray(z, dtype=np.float64)
    tx, ty = np.zeros(max(nxest, 2 * kx + 2)), np.zeros(max(nyest, 2 * ky + 2))
    c = np.zeros(max(nxest - kx - 1, kx + 1) * max(nyest - ky - 1, ky + 1))
    n, fp = np.zeros(3, np.int32), np.zeros(1)
    assert lib.hc_regrid_fit(_p(z), mx, my, kx, ky, ctypes.c_double(s), nxest, nyest, maxit, _p(tx), _p(ty), _p(c),
                             _p(n), _p(fp)) == 0
    nx, ny, ier = (int(v) for v in n)
    return nx, tx[:nx], ny, ty[:ny], c[:max(nx - kx - 1, 0) * max(ny - ky - 1, 0)], float(fp[0]), ier


def scipy_fit(z, kx, ky, s, nxest=None, nyest=None, maxit=20):
    """scipy's FITPACK regrid with RectBivariateSpline's arguments (_fitpack2._regrid_smth)."""
    from scipy.interpolate import _fitpack

    mx, my = z.shape
    x, y = np.arange(mx, dtype=float), np.arange(my, dtype=float)
    nxest = nxest or mx + kx + 1
    nyest = nyest or my + ky + 1
    lwrk = (4 + mx + my + nxest * (my + 2 * kx + 5) + nyest * (2 * ky + 5) + mx * (kx + 1) + my * (ky + 1) +
            max((nxest - kx - 1) * (nyest - ky - 1), my))
    wrk, iwrk = np.zeros(lwrk), np.zeros(3 + mx + my + nxest + nyest, np.int32)
    nx, tx, ny, ty, c, fp, ier = _fitpack.regrid(0, x, y, np.ravel(z), 0.0, mx - 1.0, 0.0, my - 1.0, kx, ky, s,
                                                 nxest, nyest, maxit, wrk, iwrk)
    return nx, tx[:nx], ny, ty[:ny], c[:(nx - kx - 1) * (ny - ky - 1)], float(fp), int(ier)


def same_fit(a, b):
    """Same ier, knot counts and knots exactly; fp within 1e-12 relative; c within 1e-10 of max |c|."""
    if a[6] != b[6] or a[0] != b[0] or a[2] != b[2]:
        return False
    if not (np.array_equal(a[1], b[1]) and np.array_equal(a[3], b[3])):
        return False
    if abs(a[5] - b[5]) > 1e-12 * max(abs(b[5]), 1e-300):
        return False
    scale = max(np.max(np.abs(b[4])), 1e-300)
    return bool(np.max(np.abs(a[4] - b[4])) <= 1e-10 * scale)


def one_axis_full(fit, z, kx, ky):
    mx, my = z.shape
    return fit[0] == mx + kx + 1 or fit[2] == my + ky + 1


def corpus(golden_cube):
    """Seeded cases: every SHAPE x degree pair with smooth + noise data at s from near interpolation (the
    ier = 3 region) to beyond fp0, constant planes, and the ten repaired golden input planes."""
    from oracle.map_img_oracle import replace_nans_with_interpolated_values

    rng = np.random.default_rng(2024)
    cases = []
    for mx, my in SHAPES:
        yy, xx = np.mgrid[0:mx, 0:my]
        for kx, ky in DEGREES:
            z = (np.sin(xx / rng.uniform(3, 12)) * np.cos(yy / rng.uniform(3, 12)) +
                 0.1 * rng.normal(size=(mx, my)))
            m = mx * my
            for f in (1e-6, 1e-3, 0.05, 0.3, 0.5, 1.0, 2.0, 3.0, 1e4):   # s / (m sigma^2); 1e4: beyond fp0
                cases.append((z, kx, ky, f * m * 0.01))
            cases.append((np.full((mx, my), rng.normal()), kx, ky, 1e-3))
    for l in range(golden_cube.shape[0]):
        plane = golden_cube[l]
        if np.all(np.isnan(plane)):
            continue
        z = replace_nans_with_interpolated_values(plane)
        for kx, ky in DEGREES:
            cases.append((z, kx, ky, 2.34))
    return cases


def test_host_fit_matches_fitpack_regrid(regrid_so, golden_arrays):
    cases = corpus(golden_arrays['inputs/test.fits/PRIMARY'])
    assert len(cases) >= 500
    mismatched, excluded, iers = [], [], {}
    for z, kx, ky, s in cases:
        a, b = host_fit(regrid_so, z, kx, ky, s), scipy_fit(z, kx, ky, s)
        iers[b[6]] = iers.get(b[6], 0) + 1
        if same_fit(a, b):
            continue
        if one_axis_full(a, z, kx, ky) or one_axis_full(b, z, kx, ky):
            excluded.append((z.shape, kx, ky, s, a[5], b[5]))
        else:
            mismatched.append((z.shape, kx, ky, s, a[6], b[6], a[0], b[0], a[2], b[2], a[5], b[5]))
    print(f'{len(cases)} cases, scipy ier counts {iers}; excluded (one axis at its interpolation knot count, '
          f'shape, kx, ky, s, fp here, fp scipy): {excluded}')
    assert not mismatched, mismatched[:5]
    assert iers.get(3, 0) >= 9 and iers.get(0, 0) >= 100 and iers.get(-2, 0) >= 50
    assert len(excluded) <= len(cases) // 10


def test_host_fit_matches_every_knot_growth_step(regrid_so):
    """Capped nxest / nyest stop FITPACK's knot growth early (ier = 1) and expose each intermediate knot set."""
    rng = np.random.default_rng(7)
    yy, xx = np.mgrid[0:64, 0:64]
    z = np.sin(xx / 9.0) * np.cos(yy / 7.0) + 0.1 * rng.normal(size=xx.shape)
    a = host_fit(regrid_so, z, 3, 3, 2.34, nxest=9, nyest=9)
    assert a[6] == 1 and list(a[1][4:-4]) == [32.0]      # the first knot: the middle of 62 interior sites
    for (kx, ky, s) in ((3, 3, 2.34), (1, 3, 2.34), (2, 2, 30.0)):
        final = scipy_fit(z, kx, ky, s)
        # caps below the interpolation knot counts (see the module docstring)
        for cap in range(2 * max(kx, ky) + 2, min(max(final[0], final[2]), 64 + min(kx, ky)) + 1):
            a = host_fit(regrid_so, z, kx, ky, s, nxest=cap, nyest=cap)
            b = scipy_fit(z, kx, ky, s, nxest=cap, nyest=cap)
            assert same_fit(a, b), (kx, ky, s, cap, a[6], b[6], a[1], b[1], a[3], b[3])
    # one axis capped alone (the other grows freely)
    for cap in range(8, 20):
        a = host_fit(regrid_so, z, 3, 3, 2.34, nxest=cap)
        b = scipy_fit(z, 3, 3, 2.34, nxest=cap)
        assert same_fit(a, b), cap


def test_host_evaluation_matches_bispeu(regrid_so):
    from scipy.interpolate import RectBivariateSpline

    rng = np.random.default_rng(3)
    z = rng.normal(size=(20, 30))
    for kx, ky in DEGREES:
        ref = RectBivariateSpline(np.arange(20), np.arange(30), z, kx=kx, ky=ky, s=450.0)
        tx, ty = (np.ascontiguousarray(t) for t in ref.get_knots())
        assert len(tx) < 20 + kx + 1 and len(ty) < 30 + ky + 1
        c = np.ascontiguousarray(ref.get_coeffs())
        x, y = rng.uniform(-2, 21, 500), rng.uniform(-2, 31, 500)
        x[:5], y[:5] = [0, 19, 19, 0, 7], [0, 29, 0, 29, 13]
        out = np.empty(500)
        assert regrid_so.hc_regrid_eval(_p(tx), len(tx), _p(ty), len(ty), _p(c), kx, ky, _p(x), _p(y),
                                        ctypes.c_int64(500), _p(out)) == 0
        want = ref.ev(x, y)
        assert np.max(np.abs(out - want)) <= 1e-12 * np.max(np.abs(want)), (kx, ky)


# ---- C entry points: argument checks before any device work ----------------------------------------
def test_regrid_entry_points_validate_arguments():
    lib = L.load_library()
    buf = np.zeros(64)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    bad, unsupported = -1, -3
    wb = lib.pm_regrid_work_bytes
    assert wb(0, 10, 7, 1, 3) == 0
    assert wb(2, 10, 7, 3, 3) > 0
    assert wb(-1, 10, 7, 1, 1) == bad and wb(1, 0, 7, 1, 1) == bad and wb(1, 10, 0, 1, 1) == bad
    for k in ((0, 1), (4, 1), (1, 5), (1, 0)):
        assert wb(1, 10, 7, *k) == unsupported, k
    fit = lib.pm_regrid_fit
    ok = (p, p, 1, 10, 7, 1, 3, 2.34, 20, p, p, p, p, p, p, p, None)
    assert fit(*ok[:2], 0, *ok[3:]) == 0                               # no planes: nothing to do
    for i, v in ((7, 0.0), (7, -1.0), (7, float('nan')), (7, float('inf')), (8, 0), (2, -1), (3, 0), (4, 0)):
        args = list(ok)
        args[i] = v
        assert fit(*args) == bad, (i, v)
    for i in (0, 1, 9, 10, 11, 12, 13, 14, 15):
        args = list(ok)
        args[i] = None
        assert fit(*args) == bad, i
    for k in ((4, 1), (1, 5), (0, 2)):
        assert fit(p, p, 1, 10, 7, *k, 2.34, 20, p, p, p, p, p, p, p, None) == unsupported
    assert fit(p, p, 1, 3, 7, 3, 1, 2.34, 20, p, p, p, p, p, p, p, None) == bad      # ny <= k_rows
    g = lib.pm_gather_regrid
    okg = [p, p, p, p, p, p, 4, 10, 7, 1, 3, 0, 4, p, p, 5, L.FLAG_PROPAGATE_NAN, p, None]
    assert g(*okg[:12], 0, *okg[13:]) == 0                            # empty range
    for i, v in ((11, -1), (12, -1), (11, 1), (15, -1), (16, 1), (16, 4)):
        args = list(okg)
        args[i] = v
        assert g(*args) == bad, (i, v)
    for i in (0, 1, 2, 3, 4, 5, 13, 14, 17):
        args = list(okg)
        args[i] = None
        assert g(*args) == bad, i
    args = list(okg)
    args[9] = 4
    assert g(*args) == unsupported


# ---- host-side rules of map_img -----------------------------------------------------------------------
@pytest.fixture
def no_device(monkeypatch):
    def boom(*a, **k):
        raise AssertionError('device work before the argument checks')

    for name in ('to_device', '_torch', 'regrid_fit', 'spline_prepare'):
        monkeypatch.setattr(L, name, boom)


@pytest.mark.parametrize('interp', [4, 5, (4, 1), (3, 5), (5, 5)])
def test_degree_4_and_5_with_smoothing_are_refused_before_device_work(bc_hst, no_device, interp):
    body = BX.BodyXY(constants=bc_hst, nx=7, ny=10)
    with pytest.raises(NotImplementedError):
        body.map_img(np.zeros((10, 7)), interpolation=interp, spline_smoothing=1.0, degree_interval=30)


def test_smoothing_routing_leaves_other_calls_alone():
    assert BX._smoothing_degrees('cubic', 0) is None
    assert BX._smoothing_degrees((1, 3), 0.0) is None
    assert BX._smoothing_degrees('nearest', 2.0) is None and BX._smoothing_degrees('smooth', 2.0) is None
    assert BX._smoothing_degrees('linear', 2.0) == (1, 1)
    assert BX._smoothing_degrees('quadratic', 1e-3) == (2, 2)
    assert BX._smoothing_degrees(3, 5.0) == (3, 3)
    assert BX._smoothing_degrees((1, 3), 2.34) == (1, 3)
    with pytest.raises(ValueError, match='s should be s >= 0.0'):
        BX._smoothing_degrees('cubic', -1.0)


def _ier3_case(regrid_so):
    """A plane on which FITPACK ends with ier = 3 (maxit reached: s too small)."""
    rng = np.random.default_rng(11)
    for _ in range(200):
        mx, my = rng.integers(8, 30, 2)
        z = rng.normal(size=(mx, my))
        s = float(mx * my * 10 ** rng.uniform(-6, -3))
        if scipy_fit(z, 3, 3, s)[6] == 3:
            return z, s
    raise AssertionError('no ier = 3 case found')


def test_failed_fit_raises_scipys_value_error(regrid_so, monkeypatch):
    from scipy.interpolate import RectBivariateSpline

    z, s = _ier3_case(regrid_so)
    assert host_fit(regrid_so, z, 3, 3, s)[6] == 3
    with pytest.raises(ValueError) as want:
        RectBivariateSpline(np.arange(z.shape[0]), np.arange(z.shape[1]), z, kx=3, ky=3, s=s)

    class Cube:
        shape = (3,) + z.shape

    def fake_fit(cube, k_rows, k_cols, s_):
        ier = np.array([0, host_fit(regrid_so, z, k_rows, k_cols, s_)[6], 2], dtype=np.int32)
        return L.RegridFit(None, None, None, None, None, None, ier, k_rows, k_cols)

    monkeypatch.setattr(L, 'regrid_fit', fake_fit)
    with pytest.raises(ValueError) as got:       # the first failing plane in plane order decides the text
        BX._fit_smoothing_splines(Cube(), 3, 3, s)
    assert str(got.value) == str(want.value)
    for shape, k in (((3, 9), (3, 1)), ((9, 3), (1, 3))):   # too few samples for the degree
        with pytest.raises(ValueError) as got_small:
            BX._fit_smoothing_splines(type('C', (), {'shape': (1,) + shape})(), *k, 1.0)
        with pytest.raises(ValueError) as want_small:
            RectBivariateSpline(np.arange(shape[0]), np.arange(shape[1]), np.zeros(shape), kx=k[0], ky=k[1], s=1.0)
        assert str(got_small.value) == str(want_small.value)
