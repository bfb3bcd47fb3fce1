"""
GPU tests through the public drop-in API (BodyXY / Observation), written to read
like the reference's own tests: tests/test_observation.py:1016-1280 (golden FITS),
tests/test_body_xy.py:267-486 (point transforms), :1087-1327 (map_img),
:1551-1988 (projections), :2120-2154 (backplane values), :2495-2607 (caches).
"""
import numpy as np
import pytest

from conftest import GOLDEN_ALT
from helpers import PLANE_NAMES, max_diff
from test_oracle_golden import (GOLDEN_TOL, LONLAT2XY, MAP_EXPECTED, MAP_EXPECTED_NO_PROPAGATE, check_body_point_literals,
                                check_radec_point_literals, frame_looking_at,
                                MAP_FILES, MAP_IMG, PROJ_CASES, WRAP, XY_COORDINATES)

pytestmark = pytest.mark.gpu
nan = np.nan


@pytest.fixture()
def obs(bc_hst, golden_arrays):
    import planetmapper_b200 as pm

    o = pm.Observation(data=golden_arrays['inputs/test.fits/PRIMARY'], constants=bc_hst)
    o.set_disc_params(2.5, 3.1, 3.9, 123.456)
    o.set_disc_method('<<<test>>>')
    return o


@pytest.fixture()
def body(bc_hst):
    import planetmapper_b200 as pm

    return pm.BodyXY(constants=bc_hst, nx=15, ny=10)


def _check(a, ref, name, label):
    assert a.shape == ref.shape and a.dtype == np.float64
    assert np.array_equal(np.isnan(a), np.isnan(ref)), f'{label} {name}: NaN mask'
    d = max_diff(a, ref, wrap=name in WRAP)
    assert d <= GOLDEN_TOL[name], f'{label} {name}: {d:.3e}'


def test_save_observation_backplanes_match_golden(obs, golden_arrays):
    assert obs.get_img_size() == (7, 10)
    for name in obs.backplanes:
        _check(obs.get_backplane_img(name), golden_arrays[f'test_nav.fits/{name}'], name, 'nav')
    for name in obs.backplanes:
        _check(obs.get_backplane_img(name, alt=GOLDEN_ALT), golden_arrays[f'test_nav_alt.fits/{name}'],
               name, 'nav-alt')
    assert obs._alt_adjustment == 0.0
    assert list(obs.backplanes) == PLANE_NAMES


def _map_kwargs(spec, alt):
    if spec[0] == 'rectangular':
        kw = dict(degree_interval=spec[1])
    else:
        kw = dict(projection=spec[0], lon=spec[1], lat=spec[2], size=spec[3])
    if alt:
        kw['alt'] = alt
    return kw


@pytest.mark.parametrize('fn', sorted(MAP_FILES))
def test_save_mapped_observation_matches_golden(obs, golden_arrays, fn):
    spec, alt, interp = MAP_FILES[fn]
    kw = _map_kwargs(spec, alt)
    mapped = obs.get_mapped_data(interp, **kw)
    ref = golden_arrays[f'{fn}/PRIMARY']
    assert mapped.shape == ref.shape
    assert np.array_equal(np.isnan(mapped), np.isnan(ref))
    ok = np.isfinite(ref)
    if interp == 'nearest':
        assert np.array_equal(mapped[ok], ref[ok])
    elif ok.any():
        assert np.max(np.abs(mapped[ok] - ref[ok]) / np.maximum(np.abs(ref[ok]), 1.0)) < 1e-8
    if f'{fn}/LON-GRAPHIC' in golden_arrays:
        for name in obs.backplanes:
            _check(obs.get_backplane_map(name, **kw), golden_arrays[f'{fn}/{name}'], name, fn)


def test_xy_conversions_known_answers(body):
    body.set_disc_params(5, 8, 3, 45)
    for xy, _radec, lonlat, _km, _ang in XY_COORDINATES:
        got = body.xy2lonlat(*xy)
        assert isinstance(got[0], float) and isinstance(got[1], float)
        assert np.allclose(got, lonlat, rtol=1e-9, atol=1e-8, equal_nan=True), (xy, got)
    xs = np.array([c[0][0] for c in XY_COORDINATES], dtype=float)
    ys = np.array([c[0][1] for c in XY_COORDINATES], dtype=float)
    lon, lat = body.xy2lonlat(xs, ys)
    assert lon.shape == xs.shape and lon.dtype == np.float64
    # broadcasting like SpiceBase._maybe_transform_as_arrays (tests/test_base.py:339-377)
    lon2, lat2 = body.xy2lonlat(xs[:, None], ys[None, :])
    assert lon2.shape == (len(xs), len(ys))
    assert np.array_equal(np.diag(lon2), lon, equal_nan=True)
    lon3, _ = body.xy2lonlat(np.array([4, 5]), 8)   # int arrays must give float outputs
    assert lon3.dtype == np.float64
    from planetmapper_b200 import NotFoundError

    with pytest.raises(NotFoundError):
        body.xy2lonlat(0, 0, not_found_nan=False)
    assert all(np.isnan(v) for v in body.xy2lonlat(np.nan, 8.0))
    # alt (tests/test_body_xy.py:409-428)
    for alt, e in [(123456.789, (134.58218536012419, 4.708273802335033)),
                   (-1000, (83.89699519490205, 21.59807910857171))]:
        got = body.xy2lonlat(7.781497231832574, 8.015145501618983, alt=alt)
        assert np.allclose(got, e, rtol=0, atol=5e-8)
    for lonlat, vis, allp in LONLAT2XY:
        if vis is not None:
            assert np.allclose(body.lonlat2xy(*lonlat), vis, rtol=0, atol=1e-9, equal_nan=True), lonlat
        assert np.allclose(body.lonlat2xy(*lonlat, not_visible_nan=False), allp, rtol=0, atol=1e-9,
                           equal_nan=True), lonlat
    # points off the surface (tests/test_body_xy.py:396-410)
    for (lon, lat, alt), e in [((42, 23.4, 0), (7.781497231832574, 8.015145501618983)),
                               ((42, 23.4, -123.456), (7.776650117803703, 8.014878507462662)),
                               ((42, 23.4, 1234.567), (7.829968623728911, 8.017815455484365)),
                               ((42, 23.4, nan), (nan, nan))]:
        got = body.lonlat2xy(lon, lat, alt=alt, not_visible_nan=False)
        assert np.allclose(got, e, rtol=0, atol=1e-9, equal_nan=True), (alt, got)
    # ray-cast visibility (sub-observer longitude is 153 deg): above the near side -> visible, above
    # the far side -> hidden, 50 000 km above a point just behind the limb -> sticks out
    assert np.all(np.isfinite(body.lonlat2xy(150.0, 0.0, alt=1234.567)))
    assert np.all(np.isnan(body.lonlat2xy(330.0, 0.0, alt=1234.567)))
    assert np.all(np.isnan(body.lonlat2xy(245.0, 0.0))) and np.all(np.isfinite(body.lonlat2xy(245.0, 0.0, alt=50000.0)))
    # planetocentric inputs: the planetocentric image of a planetographic point maps to the same pixel
    lon_c, lat_c = body.graphic2centric_lonlat(150.0, 23.4)
    assert abs(lat_c - 23.4) > 1.0 and np.all(np.isfinite(body.lonlat2xy(150.0, 23.4)))
    assert np.allclose(body.lonlat2xy(lon_c, lat_c, planetocentric=True), body.lonlat2xy(150.0, 23.4), rtol=0,
                       atol=1e-9)
    # planetocentric + altitude (body.py:1048-1056): the surface point of the planetocentric direction is
    # re-expressed against the raised spheroid, then lifted along the original spheroid's normal
    got = body.lonlat2xy(lon_c, lat_c, planetocentric=True, alt=5000.0)
    assert np.all(np.isfinite(got)) and not np.allclose(got, body.lonlat2xy(150.0, 23.4, alt=5000.0), rtol=0, atol=1e-6)
    assert np.allclose(got, body.lonlat2xy(150.0, 23.4, alt=5000.0), rtol=0, atol=0.05)


@pytest.mark.parametrize('interp', ['nearest', 'linear', 'cubic', 1, 3, (3, 3)])
def test_map_img_known_answers(body, interp):
    body.set_img_size(6, 5)
    body.set_disc_params(2.75, 1.3, 2.3, 45.678)
    key = {1: 'linear', 3: 'cubic', (3, 3): 'cubic'}.get(interp, interp)
    exp = np.array(MAP_EXPECTED[key])
    got = body.map_img(MAP_IMG, degree_interval=45, interpolation=interp)
    assert got.shape == exp.shape
    assert np.array_equal(np.isnan(got), np.isnan(exp))
    ok = np.isfinite(exp)
    if key == 'nearest':
        assert np.array_equal(got[ok], exp[ok])
    else:
        assert np.max(np.abs(got[ok] - exp[ok]) / np.abs(exp[ok])) < 5e-9
    cube = np.stack([MAP_IMG, MAP_IMG * 2 + 1])   # 3-D input (tests/test_body_xy.py:1280-1300)
    got3 = body.map_img(cube, degree_interval=45, interpolation=interp)
    assert got3.shape == (2,) + exp.shape
    assert np.array_equal(got3[0], got, equal_nan=True)


def test_map_img_options_and_errors(body):
    body.set_img_size(6, 5)
    body.set_disc_params(2.75, 1.3, 2.3, 45.678)
    got = body.map_img(MAP_IMG, degree_interval=45, propagate_nan=False)   # default: linear
    exp = np.array(MAP_EXPECTED_NO_PROPAGATE)
    assert np.array_equal(np.isnan(got), np.isnan(exp))
    ok = np.isfinite(exp)
    assert np.max(np.abs(got[ok] - exp[ok]) / np.abs(exp[ok])) < 5e-9
    all_nan = body.map_img(np.full((5, 6), nan), degree_interval=45)
    assert np.all(np.isnan(all_nan))
    with pytest.raises(ValueError):
        body.map_img(np.ones((5, 5)), degree_interval=45)
    with pytest.raises(ValueError):
        body.map_img(MAP_IMG, degree_interval=45, interpolation='<<<test>>>')
    for bad in ((1, 5), 4):
        with pytest.raises(NotImplementedError):
            body.map_img(MAP_IMG, degree_interval=45, interpolation=bad)
    # manual grid (tests/test_body_xy.py:1302-1327)
    lons = np.array([10.0, 150.0, 170.0])
    lats = np.array([-30.0, 0.0])
    man = body.map_img(MAP_IMG, projection='manual', lon_coords=lons, lat_coords=lats, interpolation='nearest')
    assert man.shape == (2, 3)


@pytest.mark.parametrize('case', range(len(PROJ_CASES)))
def test_generate_map_coordinates_known_answers(body, case):
    kind, size, lon0, lat0, elon, elat = PROJ_CASES[case]
    proj = {1: 'orthographic', 2: 'azimuthal', 3: 'azimuthal equal area'}[kind]
    lons, lats, xx, yy, _tr, info = body.generate_map_coordinates(proj, size=size, lon=lon0, lat=lat0)
    assert np.allclose(lons, np.array(elon, dtype=float), equal_nan=True)
    assert np.allclose(lats, np.array(elat, dtype=float), equal_nan=True)
    assert not lons.flags.writeable and not xx.flags.writeable
    assert info == dict(projection=proj, lon=lon0, lat=lat0, size=size, xlim=None, ylim=None)
    assert xx.shape == (size, size) and np.allclose(xx[0], np.linspace(xx[0, 0], -xx[0, 0], size))


def test_empty_and_degenerate_inputs(body, bc_hst):
    """Empty point sets, maps with no cells (xlim / ylim excluding everything, body_xy.py:2985-2998)
    and a one-pixel image go through every entry point and keep their shapes."""
    import planetmapper_b200 as pm

    e = np.array([], dtype=float)
    for out in (body.xy2lonlat(e, e), body.lonlat2xy(e, e), body.lonlat2xy(e, e, alt=10.0, planetocentric=True)):
        assert all(o.shape == (0,) and o.dtype == np.float64 for o in out)
    lon2, lat2 = body.xy2lonlat(np.zeros((0, 3)), np.zeros((1, 3)))
    assert lon2.shape == lat2.shape == (0, 3)
    kw = dict(projection='orthographic', size=5, xlim=(5, 6))
    lons, lats, xx, yy, _t, _info = body.generate_map_coordinates(**kw)
    assert lons.shape == lats.shape == xx.shape == yy.shape == (5, 0)
    assert body.get_backplane_map('EMISSION', **kw).shape == (5, 0)
    img = np.arange(150.0).reshape(10, 15)
    for interp in ('nearest', 'linear', 'cubic', 'smooth'):
        assert body.map_img(img, interpolation=interp, **kw).shape == (5, 0)
    assert body.map_img(np.stack([img, img]), degree_interval=90, ylim=(100, 200)).shape == (2, 0, 4)
    one = pm.BodyXY(constants=bc_hst)   # (nx = ny = 1 in the constructor fails in centre_disc, as in the reference)
    one.set_img_size(1, 1)
    one.set_disc_params(0.0, 0.0, 5.0, 0.0)
    lon = one.get_backplane_img('LON-GRAPHIC')
    assert lon.shape == (1, 1) and np.isfinite(lon[0, 0])
    # the disc-centre pixel: the reference's literal for it (tests/test_body_xy.py:278) - not exactly the
    # sub-observer longitude, which is evaluated at its own light time
    assert abs(lon[0, 0] - 153.1235185909613) < 1e-8 and abs(one.get_backplane_img('EMISSION')[0, 0]) < 1.0


def test_series_batches_equal_one_bodyxy_per_epoch():
    """planetmapper_b200.series: a time series in batched launches gives, frame by frame, exactly
    what a fresh BodyXY per epoch returns (the reference's only way to do a series)."""
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    prov = pm.get_default_provider()
    utcs = ['2004-12-31T2%d:%02d:00' % (h, m) for h in (1, 2) for m in (0, 20, 40)] + ['2004-12-30T03:00:00']
    ets = np.array([prov.utc2et(u) for u in utcs])
    names = ['EMISSION', 'LON-GRAPHIC', 'DOPPLER', 'RING-RADIUS']
    disc = dict(nx=40, ny=30, x0=19.5, y0=14.5, r0=12.0, rotation_radians=np.deg2rad(25.0))
    try:
        frames = S.build_series_frames('Jupiter', ets, 'EARTH', workers=2, **disc)
    finally:
        S.shutdown_pool()
    seen = 0
    for first, planes in S.iter_backplane_batches(frames, 40, 30, names, batch=3):
        got = planes.cpu().numpy()
        for k in range(got.shape[0]):
            body = pm.BodyXY('Jupiter', utcs[first + k], 'EARTH', nx=40, ny=30)
            body.set_disc_params(19.5, 14.5, 12.0, 25.0)
            ref = body.get_backplane_imgs(names)
            order = sorted(names, key=PLANE_NAMES.index)
            for j, n in enumerate(order):
                assert np.array_equal(got[k, j], ref[n], equal_nan=True), (first + k, n)
            seen += 1
    assert seen == len(utcs)


def test_map_series_equals_map_img_per_epoch():
    """series.map_series (batched x / y maps + grouped gather) gives, frame by frame, exactly what
    BodyXY(...).map_img(img_f) returns for that epoch (body_xy.py:1414-1631)."""
    import planetmapper_b200 as pm
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import series as S

    prov = pm.get_default_provider()
    utcs = ['2004-12-31T2%d:%02d:00' % (h, m) for h in (0, 1, 2) for m in (0, 30)] + ['2004-12-29T12:00:00']
    ets = np.array([prov.utc2et(u) for u in utcs])
    nx, ny = 36, 28
    disc = dict(nx=nx, ny=ny, x0=17.0, y0=13.5, r0=11.0, rotation_radians=np.deg2rad(40.0))
    frames = S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, **disc)
    rng = np.random.default_rng(11)
    imgs = rng.normal(1.0, 0.3, (len(utcs), ny, nx))
    imgs[rng.random(imgs.shape) < 0.03] = np.nan
    imgs[3] = np.nan                                         # an all-NaN image
    bodies = []
    for u in utcs:
        b = pm.BodyXY('Jupiter', u, 'EARTH', nx=nx, ny=ny)
        b.set_disc_params(17.0, 13.5, 11.0, 40.0)
        bodies.append(b)
    lons, lats, *_ = bodies[0].generate_map_coordinates(degree_interval=7.5)
    for interp in ('nearest', 'linear'):
        for prop in (True, False):
            before = L.launch_count()
            got = S.map_series(frames, imgs, nx, ny, lons, lats, interpolation=interp, propagate_nan=prop,
                               batch=4).cpu().numpy()
            launches = L.launch_count() - before
            assert got.shape == (len(utcs),) + lons.shape
            for f, b in enumerate(bodies):
                ref = b.map_img(imgs[f], interpolation=interp, propagate_nan=prop, degree_interval=7.5)
                assert np.array_equal(got[f], ref, equal_nan=True), (interp, prop, f)
            assert np.isfinite(got[0]).sum() > 100 and not np.isfinite(got[3]).any()
            if interp == 'nearest':
                assert launches == 2 * 2   # two batches x (maps + gather), not two launches per frame
    # a stack that is not a float64 CUDA tensor is converted batch by batch: float32 on the device maps as its
    # float64 copy, a host tensor as the numpy stack
    import torch
    imgs32 = torch.tensor(imgs, dtype=torch.float32, device='cuda')
    for stack, same in ((imgs32, imgs32.double()), (torch.from_numpy(imgs), imgs)):
        for interp in ('nearest', 'linear'):
            got = S.map_series(frames, stack, nx, ny, lons, lats, interpolation=interp, batch=4).cpu().numpy()
            want = S.map_series(frames, same, nx, ny, lons, lats, interpolation=interp, batch=4).cpu().numpy()
            assert np.isfinite(got).sum() > 100 and np.array_equal(got, want, equal_nan=True), (stack.dtype, interp)
    with pytest.raises(NotImplementedError):
        S.map_series(frames, imgs, nx, ny, lons, lats, interpolation='cubic')
    # the batched map kernel alone: every plane of every frame equals the single-frame call
    fd, lod, lad = L.to_device(frames), L.to_device(np.asarray(lons) % 360), L.to_device(lats)
    mask = L.mask_from_names(['PIXEL-X', 'EMISSION', 'DISTANCE', 'RING-RADIUS'])
    both = L.backplanes_map_batch(fd, lod, lad, mask).cpu().numpy()
    for f in range(len(utcs)):
        assert np.array_equal(both[f], L.backplanes_map(fd[f], lod, lad, mask).cpu().numpy(), equal_nan=True)


def test_custom_proj_strings(body):
    """Custom proj strings (body_xy.py:2970-2980): the strings the reference itself builds for its
    named projections (:2932-2968) must give exactly the named projection, and a unit-sphere
    orthographic string the textbook inverse."""
    g = body.generate_map_coordinates
    a, b = body.r_eq, body.r_polar
    for lon0, lat0 in ((0, 0), (-42, -21.3), (123.4, 90), (10, -90)):
        named = g('orthographic', lon=lon0, lat=lat0, size=41)
        proj = body.create_proj_string('ortho', to_meter=a, lon_0=lon0, lat_0=lat0,
                                       y_0=a * (b / a - 1) * np.sin(np.radians(lat0 * 2)))
        lim = max(1, b / a) * 1.01
        custom = g(proj, projection_x_coords=np.linspace(-lim, lim, 41))
        for i in range(4):
            # (xx * to_meter - x_0) / a rounds differently from xx itself: 1e-10 deg, not bitwise
            assert np.allclose(named[i], custom[i], rtol=0, atol=1e-10, equal_nan=True), (lon0, lat0, i)
        for name, pj, tm in (('azimuthal', 'aeqd', a * np.pi), ('azimuthal equal area', 'laea', a * 2)):
            named = g(name, lon=lon0, lat=lat0, size=33)
            proj = body.create_proj_string(pj, to_meter=tm, b=None, lon_0=lon0, lat_0=lat0)
            custom = g(proj, projection_x_coords=np.linspace(-1.01, 1.01, 33))
            for i in range(4):
                assert np.allclose(named[i], custom[i], rtol=0, atol=1e-10, equal_nan=True), (name, lon0, lat0, i)
    # +R=1, default origin: lon = -atan2(x, sqrt(1 - x^2 - y^2)) (west-positive axis), lat = asin(y)
    c = np.array([0, 0.25, 0.5])
    out_a = g('+proj=ortho +R=1 +axis=wnu +type=crs', projection_x_coords=c)
    out_b = g('+proj=ortho +R=1 +axis=wnu +type=crs', projection_x_coords=c, projection_y_coords=c)
    xx, yy = np.meshgrid(c, c)
    assert np.array_equal(out_a[2], xx) and np.array_equal(out_a[3], yy)
    assert np.allclose(out_a[1], np.degrees(np.arcsin(yy)), rtol=0, atol=1e-12)
    assert np.allclose(out_a[0], -np.degrees(np.arctan2(xx, np.sqrt(1 - xx**2 - yy**2))), rtol=0, atol=1e-12)
    for i in range(4):
        assert np.array_equal(out_a[i], out_b[i]) and not out_a[i].flags.writeable
    assert out_a[5]['projection_y_coords'] is None and hasattr(out_a[4], 'transform')
    # false origin and units: x_0 / y_0 in metres, to_meter scaling the user coordinates
    shifted = g('+proj=ortho +R=2 +x_0=1 +y_0=-0.5 +to_meter=4 +axis=wnu', projection_x_coords=(c * 2 + 1) / 4,
                projection_y_coords=(c * 2 - 0.5) / 4)
    assert np.allclose(shifted[0], out_a[0], rtol=0, atol=1e-12) and np.allclose(shifted[1], out_a[1], rtol=0, atol=1e-12)
    # a mapped backplane through a custom string equals the named projection's
    proj = body.create_proj_string('ortho', to_meter=a, lon_0=30, lat_0=10, y_0=a * (b / a - 1) * np.sin(np.radians(20)))
    lim = max(1, b / a) * 1.01
    m1 = body.get_backplane_map('EMISSION', projection='orthographic', lon=30, lat=10, size=21)
    m2 = body.get_backplane_map('EMISSION', projection=proj, projection_x_coords=np.linspace(-lim, lim, 21))
    assert np.allclose(m1, m2, rtol=0, atol=1e-9, equal_nan=True)


def test_map_planes_match_body_method_literals(body):
    """The scalar Body methods' 16-digit literals (reference tests/test_body.py:679, :1828-1868, :1902-1905,
    :2488-2524, :2560-2566) through get_backplane_map on a one-point manual grid."""
    names = list(body.backplanes)

    def planes_at(lon, lat):
        kw = dict(projection='manual', lon_coords=np.array([lon]), lat_coords=np.array([lat]))
        return np.array([body.get_backplane_map(n, **kw)[0, 0] for n in names])
    check_body_point_literals(planes_at)


def test_image_planes_match_body_radec_literals(bc_hst):
    """Body.ring_plane_coordinates / limb_coordinates_from_radec literals (reference tests/test_body.py:2008-2030,
    :1683-1697) through the image kernel: a one-pixel frame looking along each (ra, dec)."""
    from planetmapper_b200 import _lib as L

    check_radec_point_literals(
        lambda ra, dec: L.backplanes_img(L.to_device(frame_looking_at(bc_hst, ra, dec)[None]), 1, 1).cpu().numpy()[0, :, 0, 0])


def test_backplane_values_known_answers(body):
    """tests/test_body_xy.py:2120-2154 (8 decimals)."""
    body.set_img_size(4, 3)
    body.set_disc_params(x0=2, y0=1, r0=2, rotation=0)   # reference sets these before the check
    img = body.get_backplane_img('EMISSION')
    assert img.shape == (3, 4)
    m = body.get_backplane_map('EMISSION', degree_interval=90)
    assert m.shape == (2, 4)
    assert np.isfinite(m).all()   # emission is defined on the far side too
    assert np.nanmin(img) >= 0 and np.nanmax(img) < 90
    from planetmapper_b200 import BackplaneNotFoundError

    with pytest.raises(BackplaneNotFoundError):
        body.get_backplane('<<<test>>>')
    with pytest.raises(ValueError):
        body.register_backplane('emission', 'dup', lambda: None, lambda **k: None)


def test_cache_semantics(body):
    """Clearable vs stable caches and read-only views (tests/test_body_xy.py:2495-2590)."""
    body.set_disc_params(5, 8, 3, 45)
    a = body.get_emission_angle_img()
    assert not a.flags.writeable
    assert body.get_emission_angle_img() is a                     # cached view
    c = body.get_backplane_img('EMISSION')
    assert c.flags.writeable and c is not a and np.array_equal(c, a, equal_nan=True)
    n_stable = len(body._stable_cache)
    m = body.get_emission_angle_map(degree_interval=30)
    assert len(body._stable_cache) > n_stable
    xm = body.get_x_map(degree_interval=30)
    assert body.get_disc_method() == 'default' or isinstance(body.get_disc_method(), str)
    body.set_x0(6)                                                # clears _cache only
    assert len(body._cache) == 0
    assert body.get_emission_angle_map(degree_interval=30) is m   # stable cache survives
    xm2 = body.get_x_map(degree_interval=30)
    assert xm2 is not xm and not np.array_equal(xm, xm2, equal_nan=True)
    a2 = body.get_emission_angle_img()
    assert a2 is not a and not np.array_equal(a, a2, equal_nan=True)
    # alt is part of the key; value outside the context is restored
    b_alt = body.get_backplane_img('EMISSION', alt=1000.0)
    assert body._alt_adjustment == 0.0
    assert not np.array_equal(b_alt, a2, equal_nan=True)
    assert body.get_emission_angle_img() is a2
    with pytest.raises(ValueError):
        body.get_backplane_img('EMISSION', alt=np.inf)
    zero = type(body)(constants=body._bc)
    with pytest.raises(ValueError):
        zero.get_backplane_img('EMISSION')


def test_unsupported_options_raise(bc_hst):
    import planetmapper_b200 as pm

    for kw in (dict(aberration_correction='CN+S'), dict(observer_frame='ECLIPJ2000'),
               dict(surface_method='DSK/UNPRIORITIZED'), dict(illumination_source='JUPITER')):
        with pytest.raises(NotImplementedError):
            pm.BodyXY(constants=bc_hst, sz=5, **kw)
    b = pm.BodyXY(constants=bc_hst, sz=5)
    with pytest.raises(pm.ProjStringError):
        # proj strings outside the kernels' subset fail loudly (there is no PROJ fallback)
        b.generate_map_coordinates('+proj=moll +R=1 +axis=wnu +type=crs', projection_x_coords=np.arange(3.0))


@pytest.mark.parametrize('interp', ['nearest', 'linear', 'cubic', 'smooth', (1, 3)])
def test_mapped_data_chunked_streaming_equals_one_launch(obs, interp):
    """Observation.get_mapped_data walks the cube in wavelength chunks (the reference's plane loop,
    observation.py:892-905) when the mapped output is larger than device memory: forced here with 4-plane
    chunks on the 10-plane golden cube.  The streamed iterator (double-buffered pinned staging) and the
    chunked full result equal the single-launch result bit for bit."""
    want = obs.map_img(obs.data, interpolation=interp, degree_interval=4)     # one gather launch
    got = np.full_like(want, -7.0)
    seen = []
    for first, chunk in obs.iter_mapped_data(interp, planes_per_chunk=4, degree_interval=4):
        got[first:first + chunk.shape[0]] = chunk        # consumed before the buffer is reused
        seen.append((first, chunk.shape[0]))
    assert seen == [(0, 4), (4, 4), (8, 2)]
    assert np.array_equal(got, want, equal_nan=True)
    obs._planes_per_chunk = staticmethod(lambda src, planes_per_chunk=None, budget_bytes=None: 4)
    whole = obs.get_mapped_data(interp, degree_interval=4)
    assert whole.shape == want.shape and np.array_equal(whole, want, equal_nan=True)
    whole[0, 0, 0] = 123.0      # a copy: the cached array is untouched
    assert not np.array_equal(obs.get_mapped_data(interp, degree_interval=4), whole, equal_nan=True)


def test_backplane_getters_return_owned_arrays(body):
    """get_backplane_img / get_backplane_map hand out NEW writable float64 arrays (copies, body_xy.py:2629,
    :2663) filled by one device -> host copy; the named getters return read-only cached views."""
    a = body.get_backplane_img('EMISSION')
    b = body.get_backplane_img('EMISSION')
    assert a is not b and a.flags.writeable and a.dtype == np.float64 and a.flags.c_contiguous
    a[:] = 0.0
    assert np.array_equal(b, body.get_backplane_img('EMISSION'), equal_nan=True)
    view = body.get_emission_angle_img()
    assert not view.flags.writeable and np.array_equal(view, b, equal_nan=True)
    assert view is body.get_emission_angle_img()
    m = body.get_backplane_map('EMISSION', degree_interval=10)
    m2 = body.get_backplane_map('EMISSION', degree_interval=10)
    assert m is not m2 and m.flags.writeable and np.array_equal(m, m2, equal_nan=True)
    # single-plane requests cost one plane, a second plane escalates to its group, never the 26-plane stack
    fresh = type(body)(constants=body._bc, nx=15, ny=10)
    fresh.get_backplane_img('EMISSION')       # a surface plane brings its 12-plane stack (same intercept work)
    assert bin(fresh._cache[('img_planes_dev', 0.0)][0]).count('1') == 12
    fresh2 = type(body)(constants=body._bc, nx=15, ny=10)
    fresh2.get_backplane_img('RA')            # a lone sky plane costs one plane ...
    assert fresh2._cache[('img_planes_dev', 0.0)][0] == 1 << 4
    fresh2.get_backplane_img('RING-RADIUS')   # ... a second distinct one everything
    assert bin(fresh2._cache[('img_planes_dev', 0.0)][0]).count('1') == 26
    # read-ahead (planes >= 4 MB): every request leaves the next two planes nobody asked for in flight behind its
    # own copy; every array is handed out once, equals a direct copy, and a repeated request gets a fresh array
    big = type(body)(constants=body._bc, nx=1024, ny=600)
    one = big.get_backplane_img('EMISSION')
    state = big._cache[('img_readahead', 0.0)]
    assert sorted(state['ready']) == [PLANE_NAMES.index('LON-GRAPHIC'), PLANE_NAMES.index('LAT-GRAPHIC')]
    first = {n: big.get_backplane_img(n) for n in ('PHASE', 'LON-GRAPHIC', 'DOPPLER')}
    first['EMISSION'] = one
    assert len(state['ready']) == big._PREFETCH_WINDOW and not set(state['ready']) & state['asked']
    have, planes = big.get_backplanes_img_device(1 << 14)
    for n, arr in first.items():
        pid = PLANE_NAMES.index(n)
        direct = planes[bin(have & ((1 << pid) - 1)).count('1')].cpu().numpy()
        assert arr.flags.writeable and np.array_equal(arr, direct, equal_nan=True), n
        again = big.get_backplane_img(n)
        assert again is not arr and np.array_equal(again, arr, equal_nan=True)
    big.set_x0(500.0)      # a disc parameter change drops planes and read-ahead alike
    assert ('img_readahead', 0.0) not in big._cache
    moved = big.get_backplane_img('PHASE')
    assert not np.array_equal(moved, first['PHASE'], equal_nan=True)
    # a registered custom backplane still goes through its own getter
    body.register_backplane('custom', 'a custom plane', lambda: np.ones((10, 15)), lambda **kw: np.ones((3, 3)))
    assert np.array_equal(body.get_backplane_img('custom'), np.ones((10, 15)))


def test_progress_hook_receives_updates(obs, tmp_path):
    calls = []
    obs._set_progress_hook(lambda p, stack: calls.append((float(p), stack[-1] if stack else '')))
    obs._planes_per_chunk = staticmethod(lambda src, planes_per_chunk=None, budget_bytes=None: 4)
    obs.get_mapped_data('linear', degree_interval=10)
    mapped = [p for p, name in calls if name.endswith('_get_mapped_data')]
    assert mapped[0] == 0 and mapped[-1] == 1 and 0.4 in mapped and 0.8 in mapped    # 4 + 4 + 2 planes of 10
    calls.clear()
    obs.save_observation(str(tmp_path / 'nav.fits'), print_info=False)
    names = {name.split('.')[-1] for _, name in calls}
    assert {'save_observation', 'get_backplanes_img_device'} <= names
    obs._remove_progress_hook()
    calls.clear()
    obs.get_backplane_img('EMISSION')
    assert calls == []


def test_map_transformer_round_trips(body):
    """generate_map_coordinates' transformer slot: transform(x, y, direction='INVERSE') reproduces the lons / lats
    it came with, FORWARD maps them back onto the grid (pyproj.Transformer's interface, body_xy.py:3126)."""
    import planetmapper_b200 as pm

    for kw in (dict(projection='orthographic', lon=30, lat=-20, size=41), dict(projection='azimuthal', lat=90, size=31),
               dict(projection='azimuthal equal area', lon=-100, lat=45, size=37)):
        lons, lats, xx, yy, tr, info = body.generate_map_coordinates(**kw)
        assert isinstance(tr, pm.MapTransformer)
        lo, la = tr.transform(xx, yy, direction='INVERSE')
        ok = np.isfinite(lons)
        assert np.array_equal(np.isfinite(lo), ok) and np.all(np.isinf(lo[~ok]))     # pyproj marks failures with inf
        assert np.array_equal(lo[ok], lons[ok]) and np.array_equal(la[ok], lats[ok])
        inside = ok & (np.hypot(xx, yy) < 0.98)
        fx, fy = tr.transform(lons[inside], lats[inside])
        assert np.max(np.abs(fx - xx[inside])) < 1e-8 and np.max(np.abs(fy - yy[inside])) < 1e-8
        x1, y1 = tr.transform(float(lons[inside][0]), float(lats[inside][0]), direction='FORWARD')
        assert isinstance(x1, float) and abs(x1 - xx[inside][0]) < 1e-8
    # rectangular / manual maps are their own lon / lat system
    lons, lats, xx, yy, tr, info = body.generate_map_coordinates(degree_interval=30)
    u, v = tr.transform(lons, lats, direction='INVERSE')
    assert np.array_equal(u, lons) and np.array_equal(v, lats)
    # custom proj string with its own units
    # (+a / +b carry the body's radii in km, so "metres" are km here: to_meter = 1000 makes the user units Mm)
    proj = body.create_proj_string('ortho', lon_0=10, lat_0=20, to_meter=1000.0, x_0=5000.0, y_0=-2000.0)
    c = np.linspace(-60, 70, 25)
    lons, lats, xx, yy, tr, info = body.generate_map_coordinates(proj, projection_x_coords=c + 5, projection_y_coords=c)
    ok = np.isfinite(lons)
    assert ok.sum() > 100
    fx, fy = tr.transform(lons[ok], lats[ok])
    core = np.hypot(xx[ok] - 5, yy[ok] + 2) < 60
    assert np.max(np.abs(fx[core] - xx[ok][core])) < 1e-6 and np.max(np.abs(fy[core] - yy[ok][core])) < 1e-6
    with pytest.raises(ValueError):
        tr.transform(0.0, 0.0, direction='sideways')


def test_mapping_visible_areas_close_observer(oracle):
    """The reference's test_mapping_visible_areas (tests/test_body_xy.py:2592-2608): Jupiter seen from
    Amalthea, 2.5 radii from the centre.  The visible part of a map is exactly where the emission angle
    is <= 90 deg, for the RA map and for a mapped image alike.  (Amalthea's state comes from the synthetic
    orbit of minispice/kepler.py: the reference kernel holds it as an SPK type 17 segment.)  The image and
    map planes of the same frame are then compared with the oracle."""
    import planetmapper_b200 as pm
    from helpers import PID, check_img_planes, check_map_planes
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    body = pm.BodyXY('Jupiter', observer='amalthea', utc='2005-01-01T03:00:00', sz=10,
                     provider=KeplerOrbitProvider(pm.get_default_provider()))
    body.set_disc_params(5, 5, 3, 0)
    assert 2.0 < body.target_distance / body.r_eq < 3.0
    map_kwargs = dict(degree_interval=15)
    emission_map = body.get_backplane_map('EMISSION', **map_kwargs)
    ra_map = body.get_backplane_map('RA', **map_kwargs)
    map_img = body.map_img(np.ones((10, 10)), **map_kwargs)
    assert np.all(np.isfinite(ra_map[emission_map <= 90]))
    assert np.all(~np.isfinite(ra_map[emission_map > 90]))
    assert np.all(np.isfinite(map_img[emission_map <= 90]))
    assert np.all(~np.isfinite(map_img[emission_map > 90]))
    assert 0.15 < np.isfinite(ra_map).mean() < 0.35

    body.set_img_size(120, 90)
    body.set_disc_params(61.0, 40.5, 55.0, 200.0)
    fr = body._frame_host()
    ref, margin = oracle.backplanes_img(fr, 120, 90, with_margin=True)
    got = np.stack([body.get_backplane_img(n) for n in PLANE_NAMES])
    check_img_planes(got, ref, margin, fr, 'jupiter/amalthea', allow_epoch_quantum=True)
    lons, lats = body.generate_map_coordinates(degree_interval=5)[:2]
    refm, marginm = oracle.backplanes_map(fr, lons, lats, with_margin=True)
    gotm = np.stack([body.get_backplane_map(n, degree_interval=5) for n in PLANE_NAMES])
    check_map_planes(gotm, refm, marginm, fr, 120, 90, 'jupiter/amalthea map')
    assert np.isfinite(got[PID['EMISSION']]).sum() > 3000


def test_optimize_speed_flag(bc_hst, oracle):
    """BodyXY(optimize_speed=False) (body_xy.py:186-232, :3200-3217) runs the intercept for every pixel; with the
    reference's cut-off radius the results are identical to the default, and the header of a saved observation
    records the setting (observation.py:1330)."""
    import planetmapper_b200 as pm
    from helpers import PID, check_img_planes

    planes = {}
    for opt in (True, False):
        body = pm.BodyXY(constants=bc_hst, nx=64, ny=48, optimize_speed=opt)
        body.set_disc_params(30.0, 22.0, 18.0, 17.0)
        fr = body._frame_host()
        ref, margin = oracle.backplanes_img(fr, 64, 48, with_margin=True)
        planes[opt] = np.stack([body.get_backplane_img(n) for n in PLANE_NAMES])
        check_img_planes(planes[opt], ref, margin, fr, f'optimize_speed={opt}')
    assert np.array_equal(planes[True], planes[False], equal_nan=True)
    assert np.isfinite(planes[True][PID['EMISSION']]).sum() > 900
