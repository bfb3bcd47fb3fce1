"""
GPU parity: the CUDA kernels (through the C ABI) against the CPU oracle on the same
seeded inputs, plus size-independent properties at BASELINE.json's full sizes.

Bars (BASELINE.json north_star): on-disc masks and nearest maps bit-exact with
grazing pixels (|tangency margin| < 1e-9) excluded and counted; lon/lat/angles
<= 1e-9 deg; distances / velocities <= 1e-12 relative; linear / cubic maps <= 1e-10
relative of scipy.  Near the limb the angle bar is widened by the intercept's
conditioning number only (tests/helpers.py:surface_tolerances explains why).
"""
import numpy as np
import pytest

from helpers import (IMG_CASES, OTHER_BODIES, PID, PLANE_NAMES, WRAP, angle_diff, check_img_planes, check_map_planes,
                     img_case as _img_case, masks_equal, raw_plane_stats, surface_tolerances, write_parity_report)
from planetmapper_b200 import frame as F

pytestmark = pytest.mark.gpu

@pytest.fixture(scope='module')
def L():
    import torch

    from planetmapper_b200 import _lib

    assert torch.cuda.is_available()
    _lib.load_library()
    return _lib


@pytest.mark.parametrize('case', sorted(IMG_CASES))
def test_image_backplanes_vs_oracle(L, oracle, bc_hst, case):
    nx, ny, x0, y0, r0, rot, alt = IMG_CASES[case]
    fr = _img_case(bc_hst, nx, ny, x0, y0, r0, rot, alt)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = L.backplanes_img(L.to_device(fr[None]), nx, ny).cpu().numpy()[0]
    report, n_graz, n_mis = check_img_planes(got, ref, margin, fr, case)
    print(case, 'grazing px excluded:', n_graz, 'mask flips there:', n_mis,
          {k: round(float(v), 3) for k, v in report.items()})


def test_image_backplanes_earth_observer_saturn(L, oracle):
    """Second body / observer: Saturn (rings) from Earth, built by MiniSpice from the
    bundled extract, epoch before the SPK edge (SURVEY 8(d) C3)."""
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), 'Saturn', '2004-12-30T12:00:00', 'EARTH')
    nx = ny = 96
    fr = _img_case(bc, nx, ny, 47.5, 47.5, 18.0, 10.0)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = L.backplanes_img(L.to_device(fr[None]), nx, ny).cpu().numpy()[0]
    check_img_planes(got, ref, margin, fr, 'saturn')
    ring = got[PID['RING-RADIUS']]
    assert np.isfinite(ring).sum() > 1000 and np.nanmax(ring) > 136780  # A ring is in frame


@pytest.mark.parametrize('target,observer,nx,ny,x0,y0,r0,rot', OTHER_BODIES)
def test_other_bodies_vs_oracle(L, oracle, target, observer, nx, ny, x0, y0, r0, rot):
    """Bodies outside BASELINE.json's configs: retrograde spin, spheres, near field,
    east-positive longitudes (image and map direction)."""
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), target, '2004-12-31T00:00:00', observer)
    fr = _img_case(bc, nx, ny, x0, y0, r0, rot)
    ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
    got = L.backplanes_img(L.to_device(fr[None]), nx, ny).cpu().numpy()[0]
    check_img_planes(got, ref, margin, fr, f'{target}/{observer}', allow_epoch_quantum=True)
    lons = np.arange(2.5, 360, 5.0)[::-1]
    lats = np.arange(-87.5, 90, 5.0)
    lo, la = np.meshgrid(lons, lats)
    refm, marginm = oracle.backplanes_map(fr, lo, la, with_margin=True)
    gotm = L.backplanes_map(L.to_device(fr), L.to_device(lo), L.to_device(la)).cpu().numpy()
    check_map_planes(gotm, refm, marginm, fr, nx, ny, f'{target}/{observer} map')


@pytest.mark.parametrize('target,observer', [('Moon', 'EARTH'), ('Venus', 'EARTH'), ('Earth', 'MOON'), ('Mars', 'EARTH')])
def test_other_bodies_large_disc_limb_vs_oracle(L, oracle, target, observer):
    """The same bodies with a 700-pixel disc: thousands of limb pixels per body, so the grazing-ray
    branch of sincpt (light time iterated to convergence) is exercised on near-field, retrograde and
    east-positive geometries, all 26 planes."""
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), target, '2004-12-31T00:00:00', observer)
    sz = 768
    fr = _img_case(bc, sz, sz, 380.3, 390.7, 350.0, 33.0)
    ref, margin = oracle.backplanes_img(fr, sz, sz, with_margin=True)
    got = L.backplanes_img(L.to_device(fr[None]), sz, sz).cpu().numpy()[0]
    report, n_graz, n_mis = check_img_planes(got, ref, margin, fr, f'{target}/{observer} 768', allow_epoch_quantum=True)
    emi = ref[PID['EMISSION']]
    assert (emi > 89.1).sum() > 20, 'no grazing pixels in this frame'


def test_plane_mask_subsets_match_full_stack(L, bc_hst):
    fr = _img_case(bc_hst, 60, 50, 29.5, 24.5, 22.0, 12.0)
    fd = L.to_device(fr[None])
    full = L.backplanes_img(fd, 60, 50).cpu().numpy()[0]
    for names in (['EMISSION'], ['LON-GRAPHIC', 'LAT-GRAPHIC'], ['RA', 'DEC', 'KM-X'], ['DOPPLER'],
                  ['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE', 'DISTANCE'],
                  ['LIMB-DISTANCE'], ['LOCAL-SOLAR-TIME'], ['AZIMUTH', 'PIXEL-X']):
        mask = L.mask_from_names(names)
        sub = L.backplanes_img(fd, 60, 50, mask).cpu().numpy()[0]
        for slot, pid in enumerate(sorted(PID[n] for n in names)):
            assert np.array_equal(sub[slot], full[pid], equal_nan=True), PLANE_NAMES[pid]


@pytest.mark.parametrize('nx,ny,x0,y0', [(60, 50, 29.5, 24.5), (333, 129, 400.0, -20.0), (16, 700, 3.0, 650.0)])
def test_host_frame_launch_equals_device_frame_launch(L, bc_hst, nx, ny, x0, y0):
    """pm_backplanes_img_host (constants as a kernel parameter, derived on the host, tiles handed out from the
    disc centre outwards) gives bit-identical planes to pm_backplanes_img (frame in device memory, constants
    derived in each CTA's prologue): the derivation is exactly rounded IEEE arithmetic on both sides."""
    fr = _img_case(bc_hst, nx, ny, x0, y0, 22.0, 12.0)
    for names in (None, ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'INCIDENCE', 'EMISSION', 'PHASE',
                         'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER'],
                  ['EMISSION'], ['RA', 'RING-RADIUS', 'LIMB-DISTANCE', 'DISTANCE']):
        mask = L.ALL_PLANES if names is None else L.mask_from_names(names)
        dev = L.backplanes_img(L.to_device(fr[None]), nx, ny, mask)[0].cpu().numpy()
        host = L.backplanes_img_host(fr, nx, ny, mask).cpu().numpy()
        assert np.array_equal(dev, host, equal_nan=True), names


def test_frame_batch_equals_single_frames(L, bc_hst):
    frames = np.stack([_img_case(bc_hst, 40, 30, 19.5 + k, 14.5 - k, 12.0 + k, 7.0 * k) for k in range(5)])
    mask = L.mask_from_names(['LON-GRAPHIC', 'EMISSION', 'DISTANCE', 'RADIAL-VELOCITY'])
    batch = L.backplanes_img(L.to_device(frames), 40, 30, mask).cpu().numpy()
    for k in range(5):
        one = L.backplanes_img(L.to_device(frames[k:k + 1]), 40, 30, mask).cpu().numpy()[0]
        assert np.array_equal(batch[k], one, equal_nan=True)


def _grid(step):
    lons = np.arange(step / 2, 360, step)[::-1]
    lats = np.arange(-90 + step / 2, 90, step)
    return np.meshgrid(lons, lats)


def test_map_host_frame_and_xy_instantiation_equal_the_general_kernel(L, bc_hst):
    """pm_backplanes_map_host (kernel-parameter frame) equals pm_backplanes_map bit for bit, and the x / y map
    instantiation (plane set fixed at compile time, phase / incidence / state never computed) gives the same
    x_map / y_map bits as the general kernel asked for more planes; the batched launch too.  (The general kernel is the one compared with the oracle below.)"""
    nx, ny = 200, 160
    fr = _img_case(bc_hst, nx, ny, 101.3, 77.9, 61.0, 33.0)
    lo, la = _grid(0.75)
    lo = lo.copy()
    lo[0, 0] = np.nan
    la[1, 1] = np.inf
    lo[2, 2] = -725.0
    lod, lad, frd = L.to_device(lo), L.to_device(la), L.to_device(fr)
    xy = L.mask_from_names(['PIXEL-X', 'PIXEL-Y'])
    wide = L.mask_from_names(['PIXEL-X', 'PIXEL-Y', 'RA', 'EMISSION', 'DOPPLER'])
    ref_all = L.backplanes_map(frd, lod, lad).cpu().numpy()
    assert np.array_equal(L.backplanes_map_host(fr, lod, lad).cpu().numpy(), ref_all, equal_nan=True)
    ref_xy = ref_all[[L.PLANE_ID['PIXEL-X'], L.PLANE_ID['PIXEL-Y']]]
    assert np.isfinite(ref_xy).sum() > 10000
    for got in (L.backplanes_map(frd, lod, lad, xy), L.backplanes_map_host(fr, lod, lad, xy),
                L.backplanes_map_batch(L.to_device(np.stack([fr, fr])), lod, lad, xy)[1]):
        assert np.array_equal(got.cpu().numpy(), ref_xy, equal_nan=True)
    w = L.backplanes_map_host(fr, lod, lad, wide).cpu().numpy()
    ids = sorted(L.PLANE_ID[n] for n in ('PIXEL-X', 'PIXEL-Y', 'RA', 'EMISSION', 'DOPPLER'))
    assert np.array_equal(w, ref_all[ids], equal_nan=True)

@pytest.mark.parametrize('case', ['golden-7x10', 'rot-200x160', 'golden-7x10-alt'])
def test_map_backplanes_vs_oracle(L, oracle, bc_hst, case):
    nx, ny, x0, y0, r0, rot, alt = IMG_CASES[case]
    fr = _img_case(bc_hst, nx, ny, x0, y0, r0, rot, alt)
    lo, la = _grid(3.0)
    lo = lo.copy()
    lo[0, 0] = np.nan      # non-finite inputs -> NaN outputs
    la[1, 1] = np.inf
    lo[2, 2] = -725.0      # lon % 360
    ref, margin = oracle.backplanes_map(fr, lo, la, with_margin=True)
    got = L.backplanes_map(L.to_device(fr), L.to_device(lo), L.to_device(la)).cpu().numpy()
    check_map_planes(got, ref, margin, fr, nx, ny, case)


def test_point_transforms_vs_oracle(L, oracle, bc_hst):
    fr = _img_case(bc_hst, 15, 10, 5, 8, 3, 45)
    fd = L.to_device(fr)
    rng = np.random.default_rng(1)
    xs = np.concatenate([rng.uniform(-2, 12, 4000), [np.nan, 5.0, np.inf, 5.0]])
    ys = np.concatenate([rng.uniform(2, 14, 4000), [8.0, np.nan, 8.0, 8.0]])
    rl, rb, rmiss = oracle.xy2lonlat(fr, xs, ys)
    gl, gb, gmiss = L.xy2lonlat(fd, L.to_device(xs), L.to_device(ys))
    gl, gb = gl.cpu().numpy(), gb.cpu().numpy()
    mism = np.isnan(gl) != np.isnan(rl)
    assert mism.sum() <= 2 and abs(int(gmiss.item()) - rmiss) <= 2   # only exact-limb grazers may flip
    ok = np.isfinite(gl) & np.isfinite(rl)
    # conditioning: compare through the inverse transform instead of raw lon/lat
    assert np.nanmax(np.abs(gb[ok] - rb[ok])) < 2e-7 and np.nanmax(angle_diff(gl[ok], rl[ok])) < 2e-6
    core = ok & (np.hypot(xs - 5, ys - 8) < 2.5)   # well inside the disc (r0 = 3)
    assert np.max(np.abs(gb[core] - rb[core])) < 1e-9
    assert np.max(angle_diff(gl[core], rl[core]) * np.cos(np.deg2rad(rb[core]))) < 1e-9
    lon = np.concatenate([rng.uniform(-360, 720, 4000), [np.nan, 0.0, np.inf]])
    lat = np.concatenate([rng.uniform(-90, 90, 4000), [0.0, np.nan, 0.0]])
    for nvn in (True, False):
        rx, ry = oracle.lonlat2xy(fr, lon, lat, not_visible_nan=nvn)
        gx, gy = L.lonlat2xy(fd, L.to_device(lon), L.to_device(lat), nvn)
        gx, gy = gx.cpu().numpy(), gy.cpu().numpy()
        assert np.array_equal(np.isnan(gx), np.isnan(rx))
        ok = np.isfinite(rx)
        assert np.max(np.abs(gx[ok] - rx[ok])) < 1e-9 and np.max(np.abs(gy[ok] - ry[ok])) < 1e-9
        # points above / below the surface (ray-cast visibility, body.py:2131-2150) and
        # planetocentric inputs (spice.latsrf, body.py:2966-2982)
        for alt, pc in ((1234.5, False), (-300.0, False), (50000.0, False), (0.0, True), (2345.6, True),
                        (-150.0, True)):
            rx, ry = oracle.lonlat2xy(fr, lon, lat, not_visible_nan=nvn, alt=alt, planetocentric=pc)
            gx, gy = L.lonlat2xy(fd, L.to_device(lon), L.to_device(lat), nvn, alt=alt, planetocentric=pc)
            gx, gy = gx.cpu().numpy(), gy.cpu().numpy()
            assert (np.isnan(gx) != np.isnan(rx)).sum() <= 2, (alt, pc)   # only limb grazers may flip
            ok = np.isfinite(rx) & np.isfinite(gx)
            assert ok.sum() > 1000 or (alt < 0 and nvn)   # points below the surface are always hidden
            if ok.any():
                assert np.max(np.abs(gx[ok] - rx[ok])) < 1e-9 and np.max(np.abs(gy[ok] - ry[ok])) < 1e-9, (alt, pc)


@pytest.mark.parametrize('kind,lon0,lat0', [(1, 0, 0), (1, 123.456, -2), (1, -42, -21.3), (1, 10, 90), (1, 0, -90),
                                            (2, 0, 0), (2, 123.456, 90), (2, 12.345, 42), (2, 0, -90),
                                            (3, 0, 0), (3, 34, -12), (3, 5, 90)])
def test_projection_inverse_vs_oracle(L, oracle, bc_hst, kind, lon0, lat0):
    a, b = bc_hst.r_eq, bc_hst.r_polar
    c = np.linspace(-1.01, 1.01, 257)
    xx, yy = np.meshgrid(c, c)
    xx = xx.copy()
    xx[0, 0] = np.nan
    for sign in (-1.0, 1.0):
        rlon, rlat = oracle.proj_inverse(kind, a, b, lon0, lat0, sign, xx, yy)
        glon, glat = L.proj_inverse(kind, a, b, lon0, lat0, sign, L.to_device(xx), L.to_device(yy))
        glon, glat = glon.cpu().numpy(), glat.cpu().numpy()
        mism = np.isnan(glon) != np.isnan(rlon)
        assert mism.sum() == 0, f'{mism.sum()} mask mismatches'
        ok = np.isfinite(rlon)
        assert ok.sum() > 1000
        # near the projection edge lon/lat are ill-conditioned in x, y: compare with 1e-9
        # deg inside 99% of the disc and a conditioning-scaled bound outside
        rr = np.hypot(xx, yy)
        core = ok & (rr < 0.98)
        assert np.max(np.abs(glat[core] - rlat[core])) < 1e-9
        coslat = np.maximum(np.cos(np.deg2rad(rlat[core])), 1e-6)
        assert np.max(angle_diff(glon[core], rlon[core]) * coslat) < 1e-9
        assert np.max(np.abs(glat[ok] - rlat[ok])) < 1e-6


def _cube(rng, nl, ny, nx):
    cube = rng.normal(1.0, 0.1, (nl, ny, nx))
    cube[1, ny // 2, nx // 2] = np.nan                 # isolated NaN
    cube[2, ::3, ::2] = np.nan                         # scattered NaNs
    cube[3] = np.nan                                   # all-NaN plane
    cube[4, 2:7, 1:6] = np.nan                         # block: centre has no good neighbour
    cube[5, 0, 0] = np.inf                             # inf is repaired but not "NaN"
    cube[5, ny - 1, nx - 1] = -np.inf
    cube[6, :, :] = np.inf                             # all bad, not all NaN -> median 0
    cube[7, 1, :] = np.nan
    return cube


@pytest.mark.parametrize('nx,ny', [(12, 9), (64, 64), (5, 4)])
def test_gather_vs_scipy_oracle(L, oracle, bc_hst, nx, ny):
    from oracle import map_img_oracle as MO

    fr = _img_case(bc_hst, nx, ny, (nx - 1) / 2 + 0.3, (ny - 1) / 2 - 0.2, 0.45 * min(nx, ny), 33.0)
    lo, la = _grid(4.0)
    xy = L.backplanes_map(L.to_device(fr), L.to_device(lo), L.to_device(la),
                          L.mask_from_names(['PIXEL-X', 'PIXEL-Y']))
    xm, ym = xy[0].cpu().numpy(), xy[1].cpu().numpy()
    assert np.isfinite(xm).sum() > 50
    rng = np.random.default_rng(7)
    cube = _cube(rng, 9, ny, nx) if ny >= 9 else rng.normal(1, 0.1, (3, ny, nx))
    cd = L.to_device(cube)
    got = L.gather(cd, xy[0], xy[1], L.INTERP_NEAREST).cpu().numpy()
    ref = MO.map_img(cube, xm, ym, 'nearest')
    assert np.array_equal(got, ref, equal_nan=True), 'nearest gather must be bit-exact'
    sub = L.gather(cd, xy[0], xy[1], L.INTERP_NEAREST, plane_begin=1, plane_count=2).cpu().numpy()
    assert np.array_equal(sub, ref[1:3], equal_nan=True)
    assert np.array_equal(oracle.gather_nearest(cube, xm, ym), ref, equal_nan=True)
    mixed = [(L.INTERP_MIXED | (a << 4) | b, (a, b)) for a in (1, 2, 3) for b in (1, 2, 3) if a != b]
    for mode, name in [(L.INTERP_LINEAR, 'linear'), (L.INTERP_QUADRATIC, 'quadratic'), (L.INTERP_CUBIC, 'cubic')] + mixed:
        if (max(name) if isinstance(name, tuple) else mode) >= min(nx, ny):
            continue
        for prop in (True, False):
            spline = L.spline_prepare(cd, mode)
            got = L.gather(spline, xy[0], xy[1], mode, propagate_nan=prop).cpu().numpy()
            # the flat (unknown row length) cell order gives the same values as the 2-D grid
            flat = L.gather(spline, xy[0].reshape(-1), xy[1].reshape(-1), mode, propagate_nan=prop).cpu().numpy()
            assert np.array_equal(flat.reshape(got.shape), got, equal_nan=True), (name, prop)
            # a quad-aligned sub-range of planes equals the same planes of the full call
            if cube.shape[0] > 4:
                sub = L.gather(spline, xy[0], xy[1], mode, plane_begin=4, plane_count=3,
                               propagate_nan=prop).cpu().numpy()
                assert np.array_equal(sub, got[4:7], equal_nan=True)
            ref = MO.map_img(cube, xm, ym, name, propagate_nan=prop)
            assert np.array_equal(np.isnan(got), np.isnan(ref)), (name, prop)
            ok = np.isfinite(ref)
            scale = np.maximum(np.abs(ref[ok]), 1.0)
            rel = np.max(np.abs(got[ok] - ref[ok]) / scale)
            assert rel <= 1e-10, f'{name} propagate={prop}: rel {rel:.3e}'


@pytest.mark.parametrize('nx,ny,step,oversample,max_size', [(12, 9, 4.0, 5, 10_000), (64, 64, 4.0, 5, 10_000),
                                                             (64, 64, 2.0, 3, 150), (40, 30, 5.0, 5, 20)])
def test_smooth_vs_scipy_oracle(L, bc_hst, nx, ny, step, oversample, max_size):
    """map_img(interpolation='smooth'): PCHIP oversampling + linear against the real scipy
    PchipInterpolator / RegularGridInterpolator arranged as the reference arranges them."""
    from oracle import map_img_oracle as MO

    fr = _img_case(bc_hst, nx, ny, (nx - 1) / 2 + 0.3, (ny - 1) / 2 - 0.2, 0.4 * min(nx, ny), 33.0)
    lo, la = _grid(step)
    xy = L.backplanes_map(L.to_device(fr), L.to_device(lo), L.to_device(la),
                          L.mask_from_names(['PIXEL-X', 'PIXEL-Y']))
    xm, ym = xy[0].cpu().numpy(), xy[1].cpu().numpy()
    rng = np.random.default_rng(11)
    cube = _cube(rng, 9, ny, nx)
    cube[8, :, nx // 2] = np.nan                      # a NaN column splits every row's PCHIP
    cd = L.to_device(cube)
    for prop in (True, False):
        got = L.map_smooth(cd, xy[0], xy[1], propagate_nan=prop, oversample_by=oversample,
                           max_oversampled_img_size=max_size).cpu().numpy()
        ref = MO.map_img(cube, xm, ym, 'smooth', propagate_nan=prop, smooth_oversample_by=oversample,
                         smooth_max_oversampled_img_size=max_size)
        assert np.array_equal(np.isnan(got), np.isnan(ref)), (prop, int((np.isnan(got) != np.isnan(ref)).sum()))
        ok = np.isfinite(ref)
        assert ok.sum() > 100
        rel = np.max(np.abs(got[ok] - ref[ok]) / np.maximum(np.abs(ref[ok]), 1.0))
        assert rel <= 1e-10, f'smooth propagate={prop}: rel {rel:.3e}'


def test_nan_repair_matches_reference_recipe(L, bc_hst):
    from oracle import map_img_oracle as MO

    rng = np.random.default_rng(3)
    cube = _cube(rng, 9, 20, 17)
    spline = L.spline_prepare(L.to_device(cube), L.INTERP_LINEAR)
    coef = spline.planes().cpu().numpy()
    nanmask = spline.nanmask().cpu().numpy()
    all_nan = spline.all_nan_planes().cpu().numpy()
    for l in range(cube.shape[0]):
        assert np.array_equal(nanmask[l], np.isnan(cube[l]))
        if np.all(np.isnan(cube[l])):
            assert all_nan[l]
            continue
        assert not all_nan[l]
        ref = MO.replace_nans_with_interpolated_values(cube[l])
        assert np.allclose(coef[l], ref, rtol=1e-14, atol=0), l


def test_nan_repair_large_planes_multi_cta_median(L):
    """Time-series images are few and large: classify / nanmedian spread a plane over many CTAs
    (multi-pass radix select with global histograms).  Same recipe, same answers: odd and even
    counts of finite pixels, inf treated as bad, an isolated 3 x 3 block of NaN (median fill),
    an all-NaN plane and a plane without NaN."""
    from oracle import map_img_oracle as MO

    rng = np.random.default_rng(17)
    ny, nx = 301, 299
    # positive values over seven decades (no cancellation in the 3 x 3 means, so 1e-14 relative is meaningful)
    cube = rng.lognormal(0.0, 1.0, (5, ny, nx)) * 10.0 ** rng.integers(-3, 4, (5, ny, nx))
    cube[0][rng.random((ny, nx)) < 0.02] = np.nan
    cube[0, 100:103, 50:53] = np.nan                       # all nine neighbours bad -> nanmedian
    if np.isfinite(cube[0]).sum() % 2 == 0:
        cube[0, 0, 0] = np.nan                             # odd number of finite pixels
    cube[1][rng.random((ny, nx)) < 0.3] = np.nan
    cube[1, 5, 5] = np.inf
    if np.isfinite(cube[1]).sum() % 2 == 1:
        cube[1, 0, 0] = np.nan                             # even: mean of the two middle values
    cube[2] = np.nan
    cube[4, 7, 7] = np.nan
    cube[4, 200:203, 200:203] = np.inf
    spline = L.spline_prepare(L.to_device(cube), L.INTERP_LINEAR)
    coef = spline.planes().cpu().numpy()
    assert np.array_equal(spline.nanmask().cpu().numpy()[:5], np.isnan(cube))
    assert list(spline.all_nan_planes().cpu().numpy()[:5]) == [False, False, True, False, False]
    for l in (0, 1, 3, 4):
        ref = MO.replace_nans_with_interpolated_values(cube[l])
        assert np.array_equal(coef[l], ref) or np.allclose(coef[l], ref, rtol=1e-14, atol=0), l
        if l in (0, 4):   # the isolated block is filled with exactly np.nanmedian of the finite pixels
            r, c = (101, 51) if l == 0 else (201, 201)
            finite = cube[l][np.isfinite(cube[l])]
            assert coef[l][r, c] == np.median(finite)


# ---- size-independent properties at BASELINE.json's full sizes ------------------------
def test_full_size_2048_properties(L, bc_hst):
    """C2: 2048 x 2048, 12-plane stack (SURVEY 8(d))."""
    import torch

    sz = 2048
    fr = _img_case(bc_hst, sz, sz, (sz - 1) / 2, (sz - 1) / 2, 0.9 * (sz - 1) / 2, 0.0)
    names = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'INCIDENCE', 'EMISSION', 'PHASE',
             'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER']
    mask = L.mask_from_names(names)
    fd = L.to_device(fr[None])
    out = L.backplanes_img_host(fr, sz, sz, mask)
    again = L.backplanes_img(fd, sz, sz, mask)[0]   # device-frame launch: same bits
    assert torch.equal(torch.nan_to_num(out, nan=-1e300), torch.nan_to_num(again, nan=-1e300)), 'deterministic'
    slot = {PID[n]: i for i, n in enumerate(sorted(names, key=lambda n: PID[n]))}
    g = lambda n: out[slot[PID[n]]]
    on = torch.isfinite(g('EMISSION'))
    frac = on.double().mean().item()
    assert 0.57 < frac < 0.62   # pi 0.45^2 (r_polar / r_eq) = 59.5 % of the frame is on the disc
    for n in names:
        assert torch.equal(torch.isfinite(g(n)), on), f'{n} mask differs from EMISSION mask'
    assert g('EMISSION')[on].max().item() < 90.0 and g('EMISSION')[on].min().item() >= 0.0
    # DOPPLER is exactly the documented function of RADIAL-VELOCITY
    beta = g('RADIAL-VELOCITY')[on] / 299792.458
    assert torch.allclose(g('DOPPLER')[on], torch.sqrt((1 + beta) / (1 - beta)), rtol=1e-15, atol=0)
    # round trip xy -> lonlat -> xy through the independent inverse kernel
    ys, xs = torch.nonzero(on & (g('EMISSION') < 80.0), as_tuple=True)
    sel = torch.randperm(xs.numel(), generator=torch.Generator().manual_seed(0))[:200000].to(xs.device)
    lon, lat = g('LON-GRAPHIC')[ys[sel], xs[sel]].contiguous(), g('LAT-GRAPHIC')[ys[sel], xs[sel]].contiguous()
    x2, y2 = L.lonlat2xy(fd[0], lon, lat, True)
    assert torch.isfinite(x2).all()
    # The reference's inverse (body.py:917-948) dates the point with the sub-observer
    # light time plus a line-of-sight offset and ignores the target's translation over
    # that offset, so its own round trip is only good to ~1e-3 px at this scale (the
    # reference tests it with atol=1e-3, tests/test_body_xy.py:333-337; the CPU oracle
    # shows 1.4e-3 px on this frame).  The bar here is that inherent error, not 1e-9.
    assert (x2 - xs[sel].double()).abs().max().item() < 5e-3
    assert (y2 - ys[sel].double()).abs().max().item() < 5e-3
    # LST is a multiple of 1/3600 h
    lst = g('LOCAL-SOLAR-TIME')[on] * 3600.0
    assert (lst - torch.round(lst)).abs().max().item() < 1e-6


def test_full_size_2048_vs_oracle(L, oracle, bc_hst):
    """C2 at full size against the oracle itself (4.19 Mpix x 12 planes; the C oracle needs
    ~0.2 s on 16 threads), with the same bars as the small cases."""
    sz = 2048
    fr = _img_case(bc_hst, sz, sz, (sz - 1) / 2, (sz - 1) / 2, 0.9 * (sz - 1) / 2, 0.0)
    names = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'INCIDENCE', 'EMISSION', 'PHASE',
             'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER']
    mask = L.mask_from_names(names)   # exactly the stack BENCH times: the compile-time-mask kernel, host-frame launch
    ref_k, margin = oracle.backplanes_img(fr, sz, sz, mask, with_margin=True)
    got_k = L.backplanes_img_host(fr, sz, sz, mask).cpu().numpy()
    ids = sorted(PID[n] for n in names)
    ref = np.full((len(PLANE_NAMES), sz, sz), np.nan)
    got = np.full((len(PLANE_NAMES), sz, sz), np.nan)
    for slot, pid in enumerate(ids):
        ref[pid], got[pid] = ref_k[slot], got_k[slot]
    # raw, un-widened statistics first (written even if an assertion below fails)
    stats = raw_plane_stats(got, ref, margin, planes=names)
    stats['config'] = 'C2: Jupiter / HST 2005-01-01T00:00:00, 2048 x 2048, r0 = 0.9 (n-1)/2, GPU kernels vs CPU oracle'
    write_parity_report('C2', stats)
    report, n_graz, n_mis = check_img_planes(got, ref, margin, fr, 'C2-2048')
    on = np.isfinite(ref[PID['EMISSION']])
    assert 2.4e6 < on.sum() < 2.6e6
    print('C2 full size: grazing px excluded', n_graz, 'mask flips there', n_mis,
          {k: round(float(v), 3) for k, v in report.items()})


def test_full_size_saturn_4096_rings_vs_oracle(L, oracle):
    """C3 at full size: Saturn 4096 x 4096, ring planes + DISTANCE against the oracle."""
    import planetmapper_b200 as pm

    bc = F.build_body_constants(pm.get_default_provider(), 'Saturn', '2004-12-30T12:00:00', 'EARTH')
    sz = 4096
    fr = _img_case(bc, sz, sz, (sz - 1) / 2, (sz - 1) / 2, 800.0, 0.0)
    names = ['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE', 'DISTANCE', 'EMISSION', 'LAT-CENTRIC', 'KM-X', 'KM-Y']
    mask = L.mask_from_names(names)
    ref_k, margin = oracle.backplanes_img(fr, sz, sz, mask, with_margin=True)
    got_k = L.backplanes_img(L.to_device(fr[None]), sz, sz, mask).cpu().numpy()[0]
    ids = sorted(PID[n] for n in names)
    ref = np.full((len(PLANE_NAMES), sz, sz), np.nan)
    got = np.full((len(PLANE_NAMES), sz, sz), np.nan)
    for slot, pid in enumerate(ids):
        ref[pid], got[pid] = ref_k[slot], got_k[slot]
    stats = raw_plane_stats(got, ref, margin, planes=[n for n in names if n not in ('KM-X', 'KM-Y')])
    stats['config'] = 'C3: Saturn / EARTH 2004-12-30T12:00:00, 4096 x 4096, r0 = 800 px, GPU kernels vs CPU oracle'
    write_parity_report('C3', stats)
    check_img_planes(got, ref, margin, fr, 'C3-4096')
    ring = got[PID['RING-RADIUS']]
    assert np.isfinite(ring).sum() > 1.5e6 and np.nanmax(ring) > 136780   # the A ring is in frame


def test_very_large_frame_indexing(L, bc_hst):
    """16384 x 16384 (268 Mpix, two planes = 4.3 GB): plane offsets and pixel indices beyond 2^31
    bytes / 2^28 elements.  A window of the big frame must equal a small frame whose disc centre is
    shifted by the window origin (same rays, same arithmetic up to the rounding of x0)."""
    import torch

    sz = 16384
    names = ['EMISSION', 'LON-GRAPHIC']
    mask = L.mask_from_names(names)
    big_fr = _img_case(bc_hst, sz, sz, 8000.25, 8100.5, 7000.0, 20.0)
    big = L.backplanes_img(L.to_device(big_fr[None]), sz, sz, mask)[0]
    assert big.shape == (2, sz, sz)
    on = torch.isfinite(big[0])
    frac = float(on.double().mean())
    assert abs(frac - np.pi * 7000.0 ** 2 * (bc_hst.r_polar / bc_hst.r_eq) / sz ** 2) < 0.02    # an ellipse of that size
    for (oy, ox) in ((0, 0), (8100 - 32, 8000 - 32), (sz - 64, sz - 64), (12000, 3000), (14000, 9000)):
        small_fr = _img_case(bc_hst, 64, 64, 8000.25 - ox, 8100.5 - oy, 7000.0, 20.0)
        small = L.backplanes_img(L.to_device(small_fr[None]), 64, 64, mask)[0].cpu().numpy()
        win = big[:, oy:oy + 64, ox:ox + 64].cpu().numpy()
        assert np.array_equal(np.isnan(win), np.isnan(small)), (oy, ox)
        ok = np.isfinite(small)
        if ok.any():
            d = np.abs(win[ok] - small[ok])
            d = np.minimum(d, np.abs(d - 360.0))
            assert d.max() < 1e-7, (oy, ox, d.max())     # x0 - ox rounds differently: ~1e-12 px -> well below this
    del big


def test_full_grid_gather_properties(L, bc_hst):
    """C4 geometry: 64 x 64 cube -> 0.1 deg grid (6.48 M cells); a few planes."""
    import torch

    sz = 64
    fr = _img_case(bc_hst, sz, sz, 31.5, 31.5, 28.0, 0.0)
    lo, la = _grid(0.1)
    assert lo.shape == (1800, 3600)
    fd = L.to_device(fr)
    planes = L.backplanes_map(fd, L.to_device(lo), L.to_device(la),
                              L.mask_from_names(['PIXEL-X', 'PIXEL-Y', 'EMISSION', 'RA']))
    # packed plane order is by plane id: RA (4), PIXEL-X (6), PIXEL-Y (7), EMISSION (14)
    ra, xm, ym, emi = planes[0], planes[1], planes[2], planes[3]
    # visibility consistency (tests/test_body_xy.py:2592-2607): RA finite <=> emission < 90
    assert torch.equal(torch.isfinite(ra), emi < 90.0)
    vis = torch.isfinite(xm)
    assert 0.3 < vis.double().mean().item() < 0.5
    yy, xx = torch.meshgrid(torch.arange(sz, dtype=torch.float64, device='cuda'),
                            torch.arange(sz, dtype=torch.float64, device='cuda'), indexing='ij')
    g = torch.Generator(device='cuda').manual_seed(0)
    A = torch.randn((sz, sz), dtype=torch.float64, device='cuda', generator=g)
    B = torch.randn((sz, sz), dtype=torch.float64, device='cuda', generator=g)
    cube = torch.stack([xx, yy, A, B, 2.5 * A - 0.75 * B])
    near = L.gather(cube, xm, ym, L.INTERP_NEAREST)
    assert torch.equal(near[0][vis], torch.round(xm[vis])) and torch.equal(near[1][vis], torch.round(ym[vis]))
    assert torch.equal(torch.isfinite(near[0]), vis)
    for mode in (L.INTERP_LINEAR, L.INTERP_QUADRATIC, L.INTERP_CUBIC):
        out = L.gather(L.spline_prepare(cube, mode), xm, ym, mode, propagate_nan=True)
        if mode == L.INTERP_CUBIC:
            # sub-maps of 1799 x 40 and 1799 x 37 cells are below 20 cells per image pixel, so they run the scalar
            # kernel: this compares the 1-D DMMA path of the full grid with it (the 4 x 8 cell blocks of narrow
            # maps are tested in test_gpu_cubic_gather.py)
            xs, ys = xm[:1799, 1000:1040].contiguous(), ym[:1799, 1000:1040].contiguous()
            sub = L.gather(L.spline_prepare(cube, mode), xs, ys, mode, propagate_nan=True)
            assert torch.equal(torch.nan_to_num(sub, nan=-7.0), torch.nan_to_num(out[:, :1799, 1000:1040], nan=-7.0))
            xs, ys = xm[:1799, 1000:1037].contiguous(), ym[:1799, 1000:1037].contiguous()   # odd row length
            sub = L.gather(L.spline_prepare(cube, mode), xs, ys, mode, propagate_nan=True)
            assert torch.equal(torch.nan_to_num(sub, nan=-7.0), torch.nan_to_num(out[:, :1799, 1000:1037], nan=-7.0))
        inside = vis & (xm >= 0) & (ym >= 0) & (xm <= sz - 1) & (ym <= sz - 1)
        assert torch.equal(torch.isfinite(out[0]), inside)
        # both spline kinds reproduce linear functions: sampling the x / y ramps returns the map
        assert (out[0][inside] - xm[inside]).abs().max().item() < 1e-11
        assert (out[1][inside] - ym[inside]).abs().max().item() < 1e-11
        # linearity of the whole prepare + gather chain
        lin = 2.5 * out[2][inside] - 0.75 * out[3][inside]
        assert (out[4][inside] - lin).abs().max().item() < 1e-11


def test_c4_full_grid_gather_vs_scipy(L, oracle, bc_hst):
    """C4 at its own geometry - the configuration BENCH times: 64 x 64 planes (the bench's recipe: 1 % NaN
    pixels, plane 17 all NaN) -> the 0.1 deg grid (3600 x 1800 = 6.48 M cells), gathered in the bench's
    512-plane chunks (so the cubic DMMA kernel runs its pipelined 1-3-footprint path with plane_begin != 0
    in the second chunk) and compared with the REAL scipy (RectBivariateSpline.ev through
    oracle/map_img_oracle.map_cube_fast) on planes at chunk / quad boundaries and the all-NaN plane;
    the x / y maps themselves against the C oracle on all 6.48 M cells."""
    import torch

    from oracle import map_img_oracle as MO

    sz, nl, chunk = 64, 520, 512
    fr = _img_case(bc_hst, sz, sz, 31.5, 31.5, 28.0, 0.0)
    lo, la = _grid(0.1)
    assert lo.shape == (1800, 3600)
    xy_mask = L.mask_from_names(['PIXEL-X', 'PIXEL-Y'])
    xy = L.backplanes_map(L.to_device(fr), L.to_device(lo), L.to_device(la), xy_mask)
    xm, ym = xy[0].cpu().numpy(), xy[1].cpu().numpy()
    ref_xy, margin = oracle.backplanes_map(fr, lo, la, xy_mask, with_margin=True)
    grazing = np.where(np.isnan(margin), False, np.abs(margin) < 1e-9)
    edge = np.zeros(lo.shape, dtype=bool)   # cells within 1e-9 px of the frame edge may flip (counted)
    for v, g, n in ((ref_xy[0], xm, sz), (ref_xy[1], ym, sz)):
        w = np.where(np.isnan(v), g, v)
        with np.errstate(invalid='ignore'):
            edge |= (np.abs(w + 0.5) < 1e-9) | (np.abs(w - (n - 0.5)) < 1e-9)
    mism = (np.isnan(xm) != np.isnan(ref_xy[0])) & ~grazing & ~edge
    assert not mism.any(), int(mism.sum())
    ok = np.isfinite(xm) & np.isfinite(ref_xy[0])
    assert ok.sum() > 2.0e6
    dx, dy = np.abs(xm - ref_xy[0])[ok].max(), np.abs(ym - ref_xy[1])[ok].max()
    assert dx <= 1e-9 * sz and dy <= 1e-9 * sz, (dx, dy)     # 64 px span ~0.01 deg of sky: <= 1e-9 relative

    rng = np.random.default_rng(0)
    cube_h = rng.normal(1.0, 0.1, (nl, sz, sz))
    cube_h[rng.random((nl, sz, sz)) < 0.01] = np.nan
    cube_h[17] = np.nan
    cube = L.to_device(cube_h)
    check = [0, 3, 4, 17, 255, 256, 511, 512, 519]   # chunk and quad boundaries, the all-NaN plane
    out = torch.empty((chunk,) + lo.shape, dtype=torch.float64, device='cuda')
    report = {'cells': int(lo.size), 'visible_cells': int(np.isfinite(xm).sum()), 'planes_checked': check,
              'xy_map_max_diff_px': [float(dx), float(dy)], 'grazing_cells_excluded': int(grazing.sum()),
              'edge_cells_excluded': int(edge.sum())}
    for mode, name in ((L.INTERP_NEAREST, 'nearest'), (L.INTERP_LINEAR, 'linear'), (L.INTERP_CUBIC, 'cubic')):
        src = cube if mode == L.INTERP_NEAREST else L.spline_prepare(cube, mode)
        got = {}
        for s in range(0, nl, chunk):
            n = min(chunk, nl - s)
            L.gather(src, xy[0], xy[1], mode, plane_begin=s, plane_count=n, out=out[:n])
            for l in check:
                if s <= l < s + n:
                    got[l] = out[l - s].cpu().numpy()
        want = MO.map_cube_fast(cube_h[check], xm, ym, name)
        worst = 0.0
        for i, l in enumerate(check):
            assert np.array_equal(np.isnan(got[l]), np.isnan(want[i])), (name, l)
            if l == 17:
                assert np.isnan(got[l]).all()
                continue
            fin = np.isfinite(want[i])
            assert fin.sum() > 1.5e6, (name, l)     # propagate_nan removes the cells touching NaN pixels
            if mode == L.INTERP_NEAREST:
                assert np.array_equal(got[l][fin], want[i][fin]), (name, l)
            else:
                rel = float(np.max(np.abs(got[l][fin] - want[i][fin]) / np.maximum(np.abs(want[i][fin]), 1.0)))
                worst = max(worst, rel)
                assert rel <= 1e-10, f'{name} plane {l}: rel {rel:.3e}'
        report[name] = {'max_rel_diff_vs_scipy': worst, 'bar': 0.0 if mode == L.INTERP_NEAREST else 1e-10}
    write_parity_report('C4', report)


@pytest.mark.timeout(300, method='thread')
def test_dense_cubic_gather_any_quad_aligned_plane_range(L, bc_hst):
    """The dense-map cubic kernel works on tiles of 8 planes; a range may start on any plane quad (a cube
    sharded over ranks: 3000 planes / 2 = 1500 = 8 * 187 + 4).  Such a range used to hang the kernel (a plane
    tile straddling a 32-plane NaN word made a warp shuffle divergent).  Every quad-aligned sub-range, including
    ones that start 4 planes before a word boundary, equals the same planes of the full launch bit for bit."""
    import torch

    sz = 64
    fr = _img_case(bc_hst, sz, sz, 31.5, 31.5, 28.0, 0.0)
    lo, la = _grid(0.75)    # 115 200 cells >= 20 * 64 * 64: the DMMA kernel
    xy = L.backplanes_map(L.to_device(fr), L.to_device(lo), L.to_device(la), L.mask_from_names(['PIXEL-X', 'PIXEL-Y']))
    rng = np.random.default_rng(5)
    cube = rng.normal(1.0, 0.1, (80, sz, sz))
    cube[rng.random(cube.shape) < 0.01] = np.nan
    cube[29] = np.nan
    spline = L.spline_prepare(L.to_device(cube), L.INTERP_CUBIC)
    full = L.gather(spline, xy[0], xy[1], L.INTERP_CUBIC)
    torch.cuda.synchronize()
    for begin, count in ((4, 3), (4, 8), (12, 13), (28, 8), (28, 52), (60, 20), (36, 1), (8, 72), (76, 4)):
        sub = L.gather(spline, xy[0], xy[1], L.INTERP_CUBIC, plane_begin=begin, plane_count=count)
        torch.cuda.synchronize()
        assert torch.equal(torch.nan_to_num(sub, nan=-7.0), torch.nan_to_num(full[begin:begin + count], nan=-7.0)), (begin, count)
    # guard cells around the output are untouched (the kernel is handed a pointer 4 planes before the buffer)
    buf = torch.full((14,) + tuple(lo.shape), 5.0, dtype=torch.float64, device='cuda')
    L.gather(spline, xy[0], xy[1], L.INTERP_CUBIC, plane_begin=20, plane_count=6, out=buf[4:10])
    torch.cuda.synchronize()
    assert bool((buf[:4] == 5.0).all()) and bool((buf[10:] == 5.0).all())
    assert torch.equal(torch.nan_to_num(buf[4:10], nan=-7.0), torch.nan_to_num(full[20:26], nan=-7.0))


@pytest.mark.parametrize('kind,lon0,lat0', [(1, 0, 0), (1, 123.456, -2), (1, 10, 90), (2, 12.345, 42), (2, 0, -90),
                                            (3, 34, -12), (3, 5, 90)])
def test_projection_forward_vs_oracle(L, oracle, bc_hst, kind, lon0, lat0):
    a, b = bc_hst.r_eq, bc_hst.r_polar
    rng = np.random.default_rng(kind)
    lon = np.concatenate([rng.uniform(-360, 720, 20000), [np.nan, 0.0, np.inf, lon0 + 180.0]])
    lat = np.concatenate([rng.uniform(-90, 90, 20000), [0.0, np.nan, 0.0, -lat0]])
    for sign in (-1.0, 1.0):
        rx, ry = oracle.proj_forward(kind, a, b, lon0, lat0, sign, lon, lat)
        gx, gy = L.proj_forward(kind, a, b, lon0, lat0, sign, L.to_device(lon), L.to_device(lat))
        gx, gy = gx.cpu().numpy(), gy.cpu().numpy()
        # the visibility threshold of the orthographic projection is a floating-point comparison at the limb
        assert (np.isnan(gx) != np.isnan(rx)).sum() <= 2
        ok = np.isfinite(rx) & np.isfinite(gx)
        assert ok.sum() > 8000
        # towards the antipode the azimuthal scale c / sin(c) amplifies the last bits of acos / sin: compare
        # at 1e-12 away from it and relative to that scale near it
        with np.errstate(invalid='ignore'):
            cosc = (np.sin(np.deg2rad(lat0)) * np.sin(np.deg2rad(lat))
                    + np.cos(np.deg2rad(lat0)) * np.cos(np.deg2rad(lat)) * np.cos(np.deg2rad(lon - lon0)))
        tol = 1e-12 / np.maximum(1.0 + cosc, 1e-6) if kind != 1 else np.full(lon.shape, 1e-12)
        assert np.all(np.abs(gx[ok] - rx[ok]) <= tol[ok]) and np.all(np.abs(gy[ok] - ry[ok]) <= tol[ok])


@pytest.fixture(scope='module')
def ld_oracle(tmp_path_factory):
    import shutil

    from test_host_check import build_ld_oracle

    if not shutil.which('gcc'):
        pytest.skip('gcc not available')
    return build_ld_oracle(str(tmp_path_factory.mktemp('oracle_ld')))


@pytest.mark.parametrize('block', range(3))
def test_random_geometries_vs_extended_precision(L, oracle, ld_oracle, block):
    """The referee of tests/test_host_check.py::test_device_code_random_geometries_vs_extended_precision on
    the GPU itself: observers from 1.3 to 1e5 radii, six bodies, image and map direction - in every plane
    the kernels are as close to the 80-bit evaluation of the reference algorithm as the FP64 oracle is."""
    from helpers import assert_referee, random_geometry

    for seed in range(16 * block, 16 * block + 16):
        fr, nx, ny, label = random_geometry(seed)
        ref, margin = oracle.backplanes_img(fr, nx, ny, with_margin=True)
        assert_referee(L.backplanes_img_host(fr, nx, ny).cpu().numpy(), ref, ld_oracle(fr, nx, ny), margin, label)
        lo, la = np.meshgrid(np.arange(3.5, 360, 7.0)[::-1], np.arange(-87.5, 90, 5.0))
        refm, marginm = oracle.backplanes_map(fr, lo, la, with_margin=True)
        gotm = L.backplanes_map_host(fr, L.to_device(lo), L.to_device(la)).cpu().numpy()
        assert_referee(gotm, refm, ld_oracle(fr, nx, ny, (lo, la)), marginm, label + ' map',
                       xy_floor=1e-9 * max(nx, ny))   # 1e-9 of the frame, the bar of check_map_planes
