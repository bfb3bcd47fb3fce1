"""
Host side of the time-series point transforms (no GPU): per-epoch disc parameters of build_series_frames,
the per-epoch frames and angular tables series.transform launches with, its argument rules, and the argument
checks of the batched C entry points.
"""
import ctypes

import numpy as np
import pytest

from planetmapper_b200 import _lib as L
from planetmapper_b200 import frame as F
from planetmapper_b200 import series as S

DISC = dict(nx=64, ny=48, x0=31.5, y0=23.5, r0=20.0, rotation_radians=0.3)


def _ets(n=40):
    import planetmapper_b200 as pm

    return pm.get_default_provider().utc2et('2005-01-01T00:00:00') - 3600.0 - 60.0 * np.arange(n)[::-1]


def _disc_arrays(n):
    k = np.arange(n)
    return dict(nx=64, ny=48, x0=31.5 + 0.7 * np.sin(k), y0=23.5 - 0.1 * k, r0=20.0 + 0.05 * k,
                rotation_radians=(0.3 + 0.02 * k) % (2 * np.pi))


def test_array_disc_parameters_pack_each_epoch_serially_and_sharded():
    import planetmapper_b200 as pm

    prov = pm.get_default_provider()
    ets = _ets()
    disc = _disc_arrays(len(ets))
    serial, k2a = S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, with_km2angular=True, **disc)
    assert serial.shape == (len(ets), F.PMFRAME_NDOUBLES) and k2a.shape == (len(ets), 2, 2)
    for f in (0, 7, 23, len(ets) - 1):
        bc = F.build_body_constants(prov, 'Jupiter', None, 'EARTH', et=float(ets[f]))
        one = {k: (v[f] if isinstance(v, np.ndarray) else v) for k, v in disc.items()}
        assert np.array_equal(serial[f], F.pack_frame(bc, **one))
        assert np.array_equal(k2a[f], F.km2angular_matrix(bc))
    try:
        for workers in (2, 3):
            frames, k2a_w = S.build_series_frames('Jupiter', ets, 'EARTH', workers=workers, with_km2angular=True,
                                                  **disc)
            assert np.array_equal(frames, serial) and np.array_equal(k2a_w, k2a)
        # mixed: some parameters per epoch, others shared
        mixed = dict(disc, x0=31.5, rotation_radians=0.3)
        assert np.array_equal(S.build_series_frames('Jupiter', ets, 'EARTH', workers=2, **mixed),
                              S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, **mixed))
    finally:
        S.shutdown_pool()


def test_scalar_disc_parameters_are_unchanged():
    """Scalars broadcast: the same bits as one array of equal values per epoch, and as pack_frame per epoch."""
    import planetmapper_b200 as pm

    ets = _ets(5)
    scalar = S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, **DISC)
    arrays = {k: (np.full(len(ets), v) if k not in ('nx', 'ny') else v) for k, v in DISC.items()}
    assert np.array_equal(S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, **arrays), scalar)
    bc = F.build_body_constants(pm.get_default_provider(), 'Jupiter', None, 'EARTH', et=float(ets[3]))
    assert np.array_equal(scalar[3], F.pack_frame(bc, **DISC))


@pytest.mark.parametrize('bad', [
    dict(x0=np.zeros(3)), dict(y0=np.zeros((40, 1))), dict(r0=np.full(41, 20.0)), dict(rotation_radians=[0.1, 0.2]),
    dict(x0=np.r_[np.zeros(39), np.nan]), dict(r0=np.r_[np.inf, np.full(39, 20.0)]), dict(y0=np.nan),
    dict(rotation_radians=np.inf),
])
def test_disc_parameter_errors_before_any_worker(bad):
    S.shutdown_pool()
    with pytest.raises(ValueError):
        S.build_series_frames('Jupiter', _ets(), 'EARTH', workers=2, **dict(DISC, **bad))
    assert not S._WORKERS   # raised before a worker process was started


def test_altitude_frames_equal_pack_frame():
    """The altitude-adjusted frames series.transform launches on are BodyXY._frame_dev(alt)'s, epoch by epoch
    (Jupiter and triaxial Europa)."""
    import planetmapper_b200 as pm
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    prov = pm.get_default_provider()
    for target, p in (('Jupiter', prov), ('Europa', KeplerOrbitProvider(prov))):
        ets = _ets(3)
        disc = _disc_arrays(3)
        frames = S.build_series_frames(target, ets, 'EARTH', provider=p, **disc)
        for alt in (750.0, -1200.0, 1e-3, 34567.8912):
            adj = S.frames_at_alt(frames, alt)
            for f in range(3):
                bc = F.build_body_constants(p, target, None, 'EARTH', et=float(ets[f]))
                one = {k: (v[f] if isinstance(v, np.ndarray) else v) for k, v in disc.items()}
                assert np.array_equal(adj[f], F.pack_frame(bc, alt=alt, **one)), (target, alt, f)
        assert np.array_equal(S.frames_at_alt(frames, 0.0), frames)


def test_angular_table_rows_equal_bodyxy_angular_aux():
    """Row f: BodyXY._angular_aux of epoch f, with origin_ra / origin_dec defaulting to that epoch's target."""
    import planetmapper_b200 as pm

    prov = pm.get_default_provider()
    ets = _ets(4) + 86400.0 * np.arange(4)
    frames, k2a = S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, with_km2angular=True, **DISC)
    for kw in (dict(origin_ra=None, origin_dec=None, coordinate_rotation=12.5), dict(origin_ra=None, origin_dec=-3.0,
               coordinate_rotation=0.0), dict(origin_ra=4.25, origin_dec=None, coordinate_rotation=-90.0)):
        table = S._angular_table(frames, km2angular=k2a, **kw)
        for f, et in enumerate(ets):
            body = pm.BodyXY(constants=F.build_body_constants(prov, 'Jupiter', None, 'EARTH', et=float(et)))
            assert np.array_equal(table[f], body._angular_aux(**kw)), (kw, f)
        assert not np.array_equal(table[0], table[-1])
    assert np.isnan(S._angular_table(frames, None, None, 5.0, None)[:, 9:]).all()   # read for a km source only


def test_transform_argument_rules_need_no_device():
    frames = np.zeros((3, F.PMFRAME_NDOUBLES))
    pts = np.zeros(4)
    for args, kw in [
        (('xy', 'xy'), {}), (('centric', 'lonlat'), {}), (('xy', 'pixels'), {}), (('radec', 'radec'), {}),
        (('xy', 'radec'), dict(origin_ra=10.0)), (('lonlat', 'km'), dict(coordinate_rotation=5.0)),
        (('km', 'angular'), dict(origin_dec=1.0)),                               # needs the epochs' km2angular
        (('km', 'angular'), dict(origin_dec=1.0, km2angular=np.zeros((2, 2, 2)))),
        (('xy', 'lonlat'), dict(per_frame=True)),                                # no epoch axis of 3
        (('xy', 'lonlat'), dict(alt=np.nan)), (('radec', 'lonlat'), dict(alt=np.inf)),
        (('lonlat', 'centric'), dict(alt=-np.inf)), (('lonlat', 'lonlat'), dict(alt=np.nan, planetocentric=True)),
    ]:
        with pytest.raises(ValueError):
            S.transform(frames, *args, pts, pts, **kw)
    for bad in (np.zeros((0, F.PMFRAME_NDOUBLES)), np.zeros((3, 91)), np.zeros(F.PMFRAME_NDOUBLES)):
        with pytest.raises(ValueError):
            S.transform(bad, 'xy', 'radec', pts, pts)


# ---- C entry points: argument checks before any device work ----------------------------------------
def test_batched_entry_points_validate_arguments():
    lib = L.load_library()
    assert lib.pm_abi_version() == 10
    buf = np.zeros(4 * F.PMFRAME_NDOUBLES)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    bad, unsupported = -1, -3
    nan, inf = float('nan'), float('inf')

    x2l = lib.pm_xy2lonlat_batch            # frames, n_frames, x, y, n, stride, lon, lat, n_missed, stream
    ok = [p, 3, p, p, 4, 0, p, p, None, None]
    for i, v in ((0, None), (1, 0), (1, -2), (1, 65536), (4, -1), (5, -1), (5, 3), (5, 1 << 62)):
        args = list(ok)
        args[i] = v
        assert x2l(*args) == bad, (i, v)
    for i in (2, 3, 6, 7):
        args = list(ok)
        args[i] = None
        assert x2l(*args) == bad, i
    assert x2l(p, 3, None, None, 0, 0, None, None, None, None) == 0   # no points: nothing to do
    assert x2l(p, 3, None, None, 0, 7, None, None, None, None) == 0

    l2x = lib.pm_lonlat2xy_batch            # frames, n_frames, lon, lat, n, stride, alt, flags, x, y, stream
    ok = [p, 3, p, p, 4, 4, 0.0, L.FLAG_NOT_VISIBLE_NAN | L.FLAG_PLANETOCENTRIC, p, p, None]
    for i, v in ((0, None), (1, 0), (1, 65536), (4, -1), (5, 2), (6, nan), (6, inf), (6, -inf), (7, 8), (7, 2)):
        args = list(ok)
        args[i] = v
        assert l2x(*args) == bad, (i, v)
    for i in (2, 3, 8, 9):
        args = list(ok)
        args[i] = None
        assert l2x(*args) == bad, i
    assert l2x(p, 65535, None, None, 0, 0, 0.0, 0, None, None, None) == 0

    tr = lib.pm_transform_batch   # frames, n_frames, src, dst, a, b, n, stride, alt, flags, aux13, oa, ob, missed, st
    ok = [p, 3, 0, 3, p, p, 4, 0, 0.0, 0, None, p, p, None, None]
    for i, v in ((0, None), (1, 0), (1, 65536), (2, -1), (2, 5), (3, -1), (3, 6), (6, -1), (7, 3), (8, nan),
                 (8, inf), (9, 16)):
        args = list(ok)
        args[i] = v
        assert tr(*args) == bad, (i, v)
    for i in (4, 5, 11, 12):
        args = list(ok)
        args[i] = None
        assert tr(*args) == bad, i
    for src in (0, 1, 2, 3):
        assert tr(p, 3, src, src, p, p, 4, 0, 0.0, 0, None, p, p, None, None) == unsupported
    assert tr(p, 3, 4, 4, None, None, 0, 0, 0.0, L.FLAG_PLANETOCENTRIC, None, None, None, None, None) == 0
    assert tr(p, 3, 4, 5, None, None, 0, 9, 0.0, 0, p, None, None, None, None) == 0
