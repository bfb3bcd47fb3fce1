"""
series.iter_mapped_series (batched x / y maps, one spline preparation per batch, the grouped gather) against the
single-epoch path: every epoch of the output equals Observation(data=cube_f, ...).get_mapped_data for that epoch
bit for bit, over every interpolation mode.  Plus the dense-map cubic path, parity with scipy on a triaxial
series, the launch count per batch, and pm_gather_grouped against pm_gather_paired and pm_gather.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ('nearest', 'linear', 'quadratic', 'cubic', 1, 2, 3, (1, 3), (3, 1), (2, 3), (3, 2))
UTCS = ['2004-12-31T2%d:%02d:00' % (h, m) for h in (0, 1, 2) for m in (0, 30)] + ['2004-12-29T12:00:00']


def _jupiter_series(utcs, nx, ny, x0, y0, r0, rot_deg):
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    prov = pm.get_default_provider()
    ets = np.array([prov.utc2et(u) for u in utcs])
    return S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, nx=nx, ny=ny, x0=x0, y0=y0, r0=r0,
                                 rotation_radians=np.deg2rad(rot_deg))


def _cubes(n, nl, ny, nx, seed):
    rng = np.random.default_rng(seed)
    cubes = rng.normal(1.0, 0.3, (n, nl, ny, nx))
    cubes[rng.random(cubes.shape) < 0.03] = np.nan
    cubes[3] = np.nan              # an all-NaN epoch
    cubes[5, nl - 1] = np.nan      # an all-NaN plane
    return cubes


def _collect(it, n):
    got = None
    for first, mapped in it:
        m = mapped.cpu().numpy()
        if got is None:
            got = np.empty((n,) + m.shape[1:])
        got[first:first + len(m)] = m
    return got


def test_every_epoch_equals_get_mapped_data():
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    nx, ny = 36, 28
    k = np.arange(len(UTCS))
    x0, y0, r0, rot = 17.0 + 0.4 * np.sin(k), 13.5 - 0.3 * k, 11.0 + 0.2 * k, 40.0 + 3.0 * k
    frames = _jupiter_series(UTCS, nx, ny, x0, y0, r0, rot)
    lons, lats, *_ = pm.BodyXY('Jupiter', UTCS[0], 'EARTH', nx=nx, ny=ny).generate_map_coordinates(degree_interval=7.5)
    for nl in (1, 3, 5):
        cubes = _cubes(len(UTCS), nl, ny, nx, seed=nl)
        obs = []
        for f, u in enumerate(UTCS):
            o = pm.Observation(data=cubes[f], target='Jupiter', utc=u, observer='EARTH')
            o.set_disc_params(x0[f], y0[f], r0[f], rot[f])
            obs.append(o)
        for mode in MODES:
            for prop in (True, False):
                got = _collect(S.iter_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation=mode,
                                                    propagate_nan=prop, batch=3), len(UTCS))
                assert got.shape == (len(UTCS), nl) + lons.shape
                for f, o in enumerate(obs):
                    ref = o.get_mapped_data(mode, propagate_nan=prop, degree_interval=7.5)
                    assert np.array_equal(got[f], ref, equal_nan=True), (nl, mode, prop, f)
                assert np.isfinite(got[0]).sum() > 100 * nl and not np.isfinite(got[3]).any()
                assert not np.isfinite(got[5, nl - 1]).any()
        if nl > 1:
            continue
        # one image per epoch, 3-D input, from a CUDA tensor: (n,) + grid, equal to map_img
        import torch

        imgs = torch.from_numpy(cubes[:, 0].copy()).cuda()
        for mode in ('cubic', (2, 3)):
            got = _collect(S.iter_mapped_series(frames, imgs, nx, ny, lons, lats, interpolation=mode, batch=4),
                           len(UTCS))
            for f, o in enumerate(obs):
                ref = o.map_img(cubes[f, 0], interpolation=mode, degree_interval=7.5)
                assert np.array_equal(got[f], ref, equal_nan=True), (nl, mode, f)


def test_dense_map_cubic():
    """A 16 x 12 image onto the 1 deg grid (337 map cells per image pixel): a cube per epoch runs pm_gather's
    dense-map kernel once per epoch and equals get_mapped_data bit for bit; one image per epoch runs the grouped
    scalar kernel, whose sums differ from the dense kernel's order in the last bits only."""
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    nx, ny = 16, 12
    utcs = UTCS[:3] + UTCS[4:6] + UTCS[3:4]
    x0, y0, r0, rot = np.array([7.5, 7.2, 8.0, 7.6, 7.4, 7.0]), 5.5, 5.0, 20.0
    frames = _jupiter_series(utcs, nx, ny, x0, y0, r0, rot)
    lons, lats, *_ = pm.BodyXY('Jupiter', utcs[0], 'EARTH', nx=nx, ny=ny).generate_map_coordinates(degree_interval=1)
    assert lons.size >= 20 * nx * ny
    for nl in (4, 5, 1):
        cubes = np.random.default_rng(nl).normal(1.0, 0.3, (len(utcs), nl, ny, nx))
        cubes[1, 0, 4, 5] = np.nan
        cubes[2, nl - 1] = np.nan
        for prop in (True, False):
            got = _collect(S.iter_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation='cubic',
                                                propagate_nan=prop, batch=4), len(utcs))
            for f, u in enumerate(utcs):
                o = pm.Observation(data=cubes[f], target='Jupiter', utc=u, observer='EARTH')
                o.set_disc_params(x0[f], y0, r0, rot)
                ref = o.get_mapped_data('cubic', propagate_nan=prop, degree_interval=1)
                assert np.isfinite(ref).sum() > 1000 or (f == 2 and nl == 1)
                if nl > 1:
                    assert np.array_equal(got[f], ref, equal_nan=True), (nl, prop, f)
                else:
                    assert np.array_equal(np.isnan(got[f]), np.isnan(ref)), (nl, prop, f)
                    ok = np.isfinite(ref)
                    if ok.any():
                        assert np.max(np.abs(got[f][ok] - ref[ok])) <= 1e-12 * np.nanmax(np.abs(cubes[f])), (prop, f)


def test_triaxial_series_against_scipy(L):
    """Europa (triaxial, analytic orbit): each epoch's map equals scipy's RectBivariateSpline (oracle/
    map_img_oracle.py) through the same x / y maps to 1e-10 relative, for quadratic, cubic and mixed degrees."""
    import planetmapper_b200 as pm
    from oracle import map_img_oracle as MO
    from planetmapper_b200 import series as S
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    provider = KeplerOrbitProvider(pm.get_default_provider())
    ets = provider.utc2et('2004-12-30T00:00:00') + 60.0 * np.arange(5)
    nx, ny = 41, 37
    frames = S.build_series_frames('Europa', ets, 'EARTH', provider=provider, nx=nx, ny=ny, x0=20.0, y0=18.5,
                                   r0=15.0, rotation_radians=0.3)
    lo, la = np.meshgrid(np.arange(1.0, 360, 2.0)[::-1], np.arange(-89.0, 90, 2.0))
    xy = L.backplanes_map_batch(L.to_device(frames), L.to_device(lo % 360), L.to_device(la),
                                L.mask_from_names(['PIXEL-X', 'PIXEL-Y'])).cpu().numpy()
    yy, xx = np.mgrid[0:ny, 0:nx]
    cubes = np.stack([np.stack([np.sin(0.21 * xx + 0.1 * f) * np.cos(0.17 * yy) + 0.05 * p * xx / nx
                                for p in range(3)]) for f in range(len(ets))])
    cubes[1, 0, 10, 12] = np.nan
    cubes[2, 2, 20:22, 5:7] = np.nan
    for mode in ('quadratic', 'cubic', (1, 3), (3, 2)):
        got = _collect(S.iter_mapped_series(frames, cubes, nx, ny, lo, la, interpolation=mode, batch=2), len(ets))
        for f in range(len(ets)):
            want = MO.map_img(cubes[f], xy[f, 0], xy[f, 1], mode)
            assert np.array_equal(np.isnan(got[f]), np.isnan(want)), (mode, f)
            ok = np.isfinite(want)
            assert ok.sum() > 3 * 1000
            assert np.max(np.abs(got[f][ok] - want[ok])) <= 1e-10 * np.max(np.abs(want[ok])), (mode, f)


@pytest.fixture()
def L():
    from planetmapper_b200 import _lib

    return _lib


def test_launches_per_batch_do_not_depend_on_its_epochs(L):
    from planetmapper_b200 import series as S

    nx, ny = 30, 26
    frames = _jupiter_series(UTCS, nx, ny, 14.5, 12.5, 10.0, 15.0)
    lo, la = np.meshgrid(np.arange(2.5, 360, 5.0)[::-1], np.arange(-87.5, 90, 5.0))
    for mode, nl in (('nearest', 1), ('linear', 1), ('cubic', 1), ('cubic', 3), ((1, 2), 6)):
        counts = []
        for n in (2, 7):
            cubes = _cubes(len(UTCS), nl, ny, nx, seed=3)[:n]
            before = L.launch_count()
            batches = sum(1 for _ in S.iter_mapped_series(frames[:n], cubes, nx, ny, lo, la, interpolation=mode,
                                                          batch=n))
            counts.append(L.launch_count() - before)
            assert batches == 1
        assert counts[0] == counts[1], (mode, nl, counts)
        if mode == 'nearest':
            assert counts[0] == 2   # the maps and one gather


def test_grouped_gather_against_paired_and_single_cube_gather(L):
    """pm_gather_grouped with one plane per map equals pm_gather_paired (nearest / linear), and every group of
    every mode equals pm_gather of the same planes through the group's map, for packed (stride 1), quad
    (stride 8) and unaligned (stride 5) layouts.  37 planes, 1000 cells: neither divides the block sizes."""
    import torch

    rng = np.random.default_rng(5)
    n, ny, nx, n_cells = 37, 9, 11, 1000
    cube_h = rng.normal(0.0, 1.0, (n, ny, nx))
    cube_h[rng.random(cube_h.shape) < 0.05] = np.nan
    cube_h[7] = np.nan
    cube = torch.from_numpy(cube_h).cuda()
    maps = rng.uniform(-1.5, [nx + 0.5, ny + 0.5], (n, n_cells, 2))
    maps[rng.random((n, n_cells)) < 0.05] = np.nan
    xy = torch.from_numpy(np.ascontiguousarray(maps.transpose(0, 2, 1))).cuda()   # (n, 2, n_cells): strided maps
    modes = [L.INTERP_NEAREST, L.INTERP_LINEAR, L.INTERP_QUADRATIC, L.INTERP_CUBIC] + [
        L.INTERP_MIXED | (a << 4) | b for a in (1, 2, 3) for b in (1, 2, 3) if a != b]
    for mode in modes:
        src = cube if mode == L.INTERP_NEAREST else L.spline_prepare(cube, mode)
        for prop in (True, False):
            if mode in (L.INTERP_NEAREST, L.INTERP_LINEAR):
                paired = L.gather_paired(src, xy[:, 0], xy[:, 1], mode, propagate_nan=prop).cpu().numpy()
                grouped = L.gather_grouped(src, xy[:, 0], xy[:, 1], mode, 1, 1, propagate_nan=prop).cpu().numpy()
                assert np.array_equal(grouped[:, 0], paired, equal_nan=True), (mode, prop)
            for per_map, stride in ((1, 1), (8, 8), (3, 5), (6, 8)):
                n_maps = (n - per_map) // stride + 1
                got = L.gather_grouped(src, xy[:n_maps, 0], xy[:n_maps, 1], mode, per_map, stride,
                                       propagate_nan=prop).cpu().numpy()
                for g in range(n_maps):
                    for p in range(per_map):
                        gl = g * stride + p
                        begin = gl // 4 * 4
                        ref = L.gather(src, xy[g, 0], xy[g, 1], mode, plane_begin=begin,
                                       plane_count=min(4, n - begin), propagate_nan=prop).cpu().numpy()[gl - begin]
                        assert np.array_equal(got[g, p], ref, equal_nan=True), (mode, prop, per_map, stride, g, p)
