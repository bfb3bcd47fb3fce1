"""
GPU tests of the per-point geometry queries of Body (reference tests/test_body.py:1683-1697, :1828-1905,
:2008-2030, :2488-2524): illumination / azimuth / local solar time / distance / radial velocity at a lon / lat,
visibility of a lon / lat, and limb / ring-plane coordinates along an RA / Dec, vectorised through
pm_backplanes_map_host and pm_backplanes_points_host.
"""
import math

import numpy as np
import pytest

from helpers import IMG_CASES, PID, WRAP, check_img_planes, img_case
from test_oracle_golden import BODY_POINT_LITERALS, BODY_POINT_TOL, RADEC_POINT_LITERALS
from test_points_host import OraclePoints

pytestmark = pytest.mark.gpu

LONLAT_PLANES = {   # method -> planes it returns, in order
    'illumination_angles_from_lonlat': ['PHASE', 'INCIDENCE', 'EMISSION'],
    'azimuth_angle_from_lonlat': ['AZIMUTH'],
    'distance_from_lonlat': ['DISTANCE'],
    'radial_velocity_from_lonlat': ['RADIAL-VELOCITY'],
}
RADEC_PLANES = {
    'limb_coordinates_from_radec': ['LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC', 'LIMB-DISTANCE'],
    'ring_plane_coordinates': ['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE'],
}


@pytest.fixture()
def body(bc_hst):
    import planetmapper_b200 as pm

    return pm.BodyXY(constants=bc_hst)   # no image size, like a plain Body


def _as_tuple(v):
    return v if isinstance(v, tuple) else (v,)


def _lonlat_values(body, lon, lat):
    """plane name -> value of every lon / lat method at one point (scalar calls)."""
    out = {}
    for method, names in LONLAT_PLANES.items():
        vals = _as_tuple(getattr(body, method)(lon, lat))
        assert all(type(v) is float for v in vals), method
        out.update(zip(names, vals))
    lst = body.local_solar_time_from_lon(lon)
    assert type(lst) is float
    out['LOCAL-SOLAR-TIME'] = lst
    return out


def test_body_point_literals_through_the_methods(body):
    """Every literal of BODY_POINT_LITERALS the lon / lat methods return, scalar calls, the tolerances of
    test_oracle_golden.check_body_point_literals."""
    n_checked = 0
    for (lon, lat), expected in BODY_POINT_LITERALS:
        got = _lonlat_values(body, lon, lat)
        for name, value in expected.items():
            if name not in got:
                continue     # RA / DEC / centric literals belong to the transforms
            g = got[name]
            if name == 'LOCAL-SOLAR-TIME':
                assert abs(g - value) < 1e-12, (lon, lat, g, value)
                total = round(value * 3600)
                text = '%02d:%02d:%02d' % (total // 3600, total % 3600 // 60, total % 60)
                assert body.local_solar_time_string_from_lon(lon) == text
            else:
                assert abs(g - value) <= BODY_POINT_TOL[name], (lon, lat, name, g, value)
            n_checked += 1
    assert n_checked == 16
    assert body.local_solar_time_string_from_lon(0.0) == '22:53:47'


def test_radec_point_literals_through_the_methods(body):
    """Every entry of RADEC_POINT_LITERALS through limb_coordinates_from_radec / ring_plane_coordinates (scalar
    calls), including the NaN of the ring point behind the disc, at the tolerances of
    test_oracle_golden.check_radec_point_literals."""
    n_checked = 0
    for (ra, dec), expected in RADEC_POINT_LITERALS:
        got = {}
        for method, names in RADEC_PLANES.items():
            vals = getattr(body, method)(ra, dec)
            assert isinstance(vals, tuple) and all(type(v) is float for v in vals)
            got.update(zip(names, vals))
        for name, value in expected.items():
            g = got[name]
            n_checked += 1
            if value != value:
                assert g != g, (ra, dec, name, g)
                continue
            tol = {'RING-RADIUS': 1e-9 * abs(value), 'RING-DISTANCE': 1e-11 * abs(value), 'LIMB-DISTANCE': 1e-5}.get(
                name, 1e-7)
            d = abs(g - value)
            if name in WRAP:
                d = min(d, abs(d - 360.0))
            assert d <= tol, (ra, dec, name, g, value, d)
    assert n_checked == 19


def test_hidden_ring_point_with_only_visible_false(body):
    """The ring point behind the disc is NaN by default; with only_visible=False it is finite and farther from
    the observer than the body's surface along the same ray."""
    hidden = [rd for rd, exp in RADEC_POINT_LITERALS if len(exp) == 3 and all(v != v for v in exp.values())]
    assert hidden
    for ra, dec in hidden:
        assert all(math.isnan(v) for v in body.ring_plane_coordinates(ra, dec))
        radius, lon, dist = body.ring_plane_coordinates(ra, dec, only_visible=False)
        assert all(math.isfinite(v) for v in (radius, lon, dist))
        s_lon, s_lat = body.radec2lonlat(ra, dec)
        surface = body.distance_from_lonlat(s_lon, s_lat)
        assert math.isfinite(surface) and dist > surface, (dist, surface)


def test_points_kernel_equals_the_image_kernel_bit_for_bit(bc_hst):
    """pm_backplanes_points_host at every integer (x, y) of a 64 x 48 frame, in shuffled order, all 26 planes,
    equals pm_backplanes_img_host bit for bit, NaNs included."""
    from planetmapper_b200 import _lib as L

    nx, ny, *rest = IMG_CASES['offset-disc-partly-outside']
    fr = img_case(bc_hst, nx, ny, *rest)
    want = L.backplanes_img_host(fr, nx, ny, L.ALL_PLANES).cpu().numpy().reshape(L.N_PLANES, -1)
    order = np.random.default_rng(3).permutation(nx * ny)
    x, y = (order % nx).astype(float), (order // nx).astype(float)
    got = L.backplanes_points_host(fr, L.to_device(x), L.to_device(y), L.ALL_PLANES).cpu().numpy()
    assert np.array_equal(got.view(np.int64), want[:, order].view(np.int64))
    # a plane subset selects the same values
    sub = L.mask_from_names(['EMISSION', 'RING-RADIUS', 'PIXEL-Y'])
    got_sub = L.backplanes_points_host(fr, L.to_device(x), L.to_device(y), sub).cpu().numpy()
    rows = [PID['PIXEL-Y'], PID['EMISSION'], PID['RING-RADIUS']]
    assert np.array_equal(got_sub.view(np.int64), want[rows][:, order].view(np.int64))


def test_lonlat_methods_equal_the_map_kernel_bit_for_bit(bc_hst):
    """The lon / lat methods on the flattened cells of a 100 x 100 manual grid equal get_backplane_map's planes
    of that grid bit for bit."""
    import planetmapper_b200 as pm

    body = pm.BodyXY(constants=bc_hst, nx=64, ny=48)
    rng = np.random.default_rng(11)
    lons, lats = rng.uniform(0, 360, (100, 100)), rng.uniform(-90, 90, (100, 100))
    kw = dict(projection='manual', lon_coords=lons, lat_coords=lats)
    lo, la = lons.ravel(), lats.ravel()
    for method, names in LONLAT_PLANES.items():
        vals = _as_tuple(getattr(body, method)(lo, la))
        for name, v in zip(names, vals):
            want = body.get_backplane_map(name, **kw).ravel()
            assert v.dtype == np.float64 and v.shape == lo.shape
            assert np.array_equal(v.view(np.int64), want.view(np.int64)), (method, name)
    lst = body.local_solar_time_from_lon(lo)
    assert np.array_equal(lst.view(np.int64), body.get_backplane_map('LOCAL-SOLAR-TIME', **kw).ravel().view(np.int64))


@pytest.mark.parametrize('case', ['offset-disc-partly-outside', 'rot-200x160', 'golden-7x10-alt'])
def test_subpixel_points_match_the_oracle(oracle, bc_hst, case):
    """Random sub-pixel positions, in and outside the frame and around the limb, against the oracle's pixel code
    at the same positions, within helpers.check_img_planes's bars; the unhidden ring planes (PM_FLAG_RING_ALL)
    against the oracle's ring_coordinates along the same RA / Dec."""
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import frame as F

    nx, ny, x0, y0, r0, rot, alt = IMG_CASES[case]
    fr = img_case(bc_hst, nx, ny, x0, y0, r0, rot, alt)
    rng = np.random.default_rng(5)
    t = rng.uniform(0, 2 * np.pi, 400)
    rr = r0 * rng.uniform(0.97, 1.03, 400)
    x = np.concatenate([rng.uniform(-5, nx + 5, 600), x0 + rr * np.cos(t)])
    y = np.concatenate([rng.uniform(-5, ny + 5, 600), y0 + rr * np.sin(t)])
    got = L.backplanes_points_host(fr, L.to_device(x), L.to_device(y), L.ALL_PLANES).cpu().numpy()
    ref, margin = OraclePoints.backplanes_points(fr, x, y, with_margin=True)
    assert np.isfinite(ref[PID['EMISSION']]).sum() > 100 and np.isnan(ref[PID['EMISSION']]).sum() > 100
    check_img_planes(got, ref, margin, fr, case)

    ra, dec, _ = oracle.transform(fr, 'xy', 'radec', x, y)
    ring = L.mask_from_names(['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE'])
    g_rad, g_lon, g_dist = L.backplanes_points_host(fr, L.to_device(x), L.to_device(y), ring,
                                                    ring_all=True).cpu().numpy()
    rad, lon, dist = OraclePoints.ring_coordinates(fr, ra, dec)
    assert np.array_equal(np.isnan(g_rad), np.isnan(rad)) and np.isfinite(rad).sum() > 100
    assert np.isfinite(g_rad[np.isnan(got[PID['RING-RADIUS']])]).any()   # hidden points are kept
    p0 = float(np.linalg.norm(F.frame_field(fr, 'P0')))
    ok = np.isfinite(rad)
    assert np.max(np.abs(g_rad[ok] - rad[ok])) <= 50e-12 * p0
    assert np.max(np.abs(g_dist[ok] - dist[ok])) <= 50e-12 * p0
    stretch = dist[ok] / F.frame_field(fr, 'ring_c')[0]
    bar = np.maximum(1e-9, np.rad2deg(8 * np.spacing(p0) * stretch / np.maximum(np.abs(rad[ok]), 1.0)))
    d = np.abs(g_lon[ok] - lon[ok])
    assert np.all(np.minimum(d, 360 - d) <= bar)


def test_vectorised_calls(body):
    """10^6 points in one call: the broadcast shape, exactly the values of scalar calls at 100 sampled points,
    one launch per lon / lat method and two per RA / Dec method."""
    from planetmapper_b200 import _lib as L

    rng = np.random.default_rng(2)
    n = 10 ** 6
    lon = rng.uniform(0, 360, (1000, 1000))
    lat = rng.uniform(-90, 90, (1, 1000))          # broadcast against lon
    ra = body.target_ra + rng.uniform(-20, 20, (1000, 1000)) / 3600
    dec = body.target_dec + rng.uniform(-20, 20, (1000, 1))
    sample = rng.integers(0, n, 100)
    calls = [(m, (lon, lat), 1) for m in LONLAT_PLANES] + [('local_solar_time_from_lon', (lon,), 1)] + \
            [(m, (ra, dec), 2) for m in RADEC_PLANES]
    for method, args, launches in calls:
        fn = getattr(body, method)
        before = L.launch_count()
        vals = _as_tuple(fn(*args))
        assert L.launch_count() - before == launches, method
        for v in vals:
            assert isinstance(v, np.ndarray) and v.dtype == np.float64 and v.shape == (1000, 1000), method
        for i in sample:
            r, c = divmod(int(i), 1000)
            one = _as_tuple(fn(*(np.broadcast_to(a, (1000, 1000))[r, c] for a in args)))
            for v, s in zip(vals, one):
                assert np.array_equal(v[r, c], s, equal_nan=True), (method, r, c)
    before = L.launch_count()
    strings = body.local_solar_time_string_from_lon(lon)
    assert L.launch_count() - before == 1 and strings.dtype == np.dtype('<U8') and strings.shape == (1000, 1000)
    vis = body.test_if_lonlat_visible(lon, lat)
    assert vis.dtype == bool and vis.shape == (1000, 1000)


def test_nonfinite_inputs(body, bc_hst):
    """NaN / +-inf points give NaN (False for visibility) without disturbing their neighbours."""
    from planetmapper_b200 import _lib as L

    nan, inf = np.nan, np.inf
    lon = np.array([10.0, nan, 200.0, inf, 33.0, -inf, 153.0])
    lat = np.array([-5.0, 0.0, nan, 0.0, 20.0, 0.0, -3.0])
    bad = ~(np.isfinite(lon) & np.isfinite(lat))
    for method in LONLAT_PLANES:
        full = _as_tuple(getattr(body, method)(lon, lat))
        for k, v in enumerate(full):
            assert np.isnan(v[bad]).all(), method
            for i in np.flatnonzero(~bad):
                assert np.array_equal(v[i], _as_tuple(getattr(body, method)(lon[i], lat[i]))[k], equal_nan=True)
    vis = body.test_if_lonlat_visible(lon, lat)
    assert not vis[bad].any() and vis[-1]
    ra0, dec0 = body.target_ra, body.target_dec
    ra = np.array([ra0, nan, ra0 + 5e-3, inf, ra0, ra0 - 2e-3])
    dec = np.array([dec0, dec0, -inf, dec0, nan, dec0 + 1e-3])
    bad = ~(np.isfinite(ra) & np.isfinite(dec))
    for method in RADEC_PLANES:
        for only in (((), (False,)) if method == 'ring_plane_coordinates' else ((),)):
            full = getattr(body, method)(ra, dec, *only)
            for k, v in enumerate(full):
                assert np.isnan(v[bad]).all(), method
                for i in np.flatnonzero(~bad):
                    assert np.array_equal(v[i], getattr(body, method)(ra[i], dec[i], *only)[k], equal_nan=True)
    # the points kernel itself: non-finite x / y give NaN planes, PIXEL-X / PIXEL-Y echo the input
    nx, ny, *rest = IMG_CASES['offset-disc-partly-outside']
    fr = img_case(bc_hst, nx, ny, *rest)
    x = np.array([50.0, nan, 50.0, inf, -inf, 40.0])
    y = np.array([10.0, 10.0, nan, 10.0, 12.0, -inf])
    for ring_all in (False, True):
        out = L.backplanes_points_host(fr, L.to_device(x), L.to_device(y), L.ALL_PLANES,
                                       ring_all=ring_all).cpu().numpy()
        for k in range(L.N_PLANES):
            if k in (PID['PIXEL-X'], PID['PIXEL-Y']):
                assert np.array_equal(out[k], x if k == PID['PIXEL-X'] else y, equal_nan=True)
            else:
                assert np.isnan(out[k][1:]).all(), k
        assert np.isfinite(out[PID['EMISSION']][0])


def test_methods_work_without_an_image_size(bc_hst):
    """BodyXY(constants=...) with no image size answers every point query, like a plain Body."""
    import planetmapper_b200 as pm

    b = pm.BodyXY(constants=bc_hst)
    assert b.get_img_size() == (0, 0)
    assert all(math.isfinite(v) for v in b.illumination_angles_from_lonlat(153.0, -3.0))
    assert math.isfinite(b.azimuth_angle_from_lonlat(153.0, -3.0))
    assert math.isfinite(b.distance_from_lonlat(153.0, -3.0))
    assert math.isfinite(b.radial_velocity_from_lonlat(153.0, -3.0))
    assert isinstance(b.local_solar_time_string_from_lon(153.0), str)
    assert b.test_if_lonlat_visible(153.0, -3.0) is True
    assert b.test_if_lonlat_visible(333.0, 3.0) is False
    assert all(math.isfinite(v) for v in b.limb_coordinates_from_radec(196.3, -5.5))
    assert all(math.isfinite(v) for v in b.ring_plane_coordinates(196.3, -5.5))
    # nothing is cached: only the device frame of the transforms
    assert all(k[0] == 'frame_dev' for k in b._cache if isinstance(k, tuple))


@pytest.mark.parametrize('alt', [0.0, 1000.0])
def test_visibility_matches_the_oracle(oracle, bc_hst, alt):
    """test_if_lonlat_visible on 10^4 random points against the oracle's lon / lat -> RA / Dec with
    not_visible_nan; points within 1e-9 of grazing are excluded and counted.  At alt = 0 it is also
    emission < 90 deg."""
    import planetmapper_b200 as pm

    b = pm.BodyXY(constants=bc_hst)
    rng = np.random.default_rng(8 + int(alt))
    lon = rng.uniform(0, 360, 10 ** 4)
    lat = np.degrees(np.arcsin(rng.uniform(-1, 1, 10 ** 4)))
    vis = b.test_if_lonlat_visible(lon, lat, alt)
    assert vis.dtype == bool and vis.shape == lon.shape
    fr = b._frame_host()

    def oracle_visible(lo, la):
        ra, dec, _ = oracle.transform(fr, 'lonlat', 'radec', lo, la, alt=alt, not_visible_nan=True)
        return np.isfinite(ra) & np.isfinite(dec)

    want = oracle_visible(lon, lat)
    # grazing: the oracle's answer changes within 1e-9 deg of the point
    grazing = np.zeros(lon.shape, bool)
    for dlo, dla in ((1e-9, 0), (-1e-9, 0), (0, 1e-9), (0, -1e-9)):
        grazing |= oracle_visible(lon + dlo, np.clip(lat + dla, -90, 90)) != want
    mism = (vis != want) & ~grazing
    assert not mism.any(), f'{int(mism.sum())} visibility mismatches ({int(grazing.sum())} grazing excluded)'
    print(f'alt={alt}: {int(grazing.sum())} of {lon.size} points within 1e-9 deg of grazing excluded')
    assert 0.3 < vis.mean() < 0.7
    if alt == 0.0:
        _, _, e = b.illumination_angles_from_lonlat(lon, lat)
        assert np.array_equal(vis[~grazing], (e < 90.0)[~grazing])
