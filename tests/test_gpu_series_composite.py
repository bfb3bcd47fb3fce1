"""
series.composite_mapped_series against the fold, in numpy, of what the series API already produces: every epoch's
iter_mapped_series output and its EMISSION map (pm_backplanes_map_batch), combined by a Python loop over the epochs in
order.  Plus independence of the batch size, a mosaic of dithers of one epoch, the dense-map cubic path, the launch
count per batch and the peak device memory of a cube composite.
"""
import numpy as np
import pytest

from test_gpu_series_map import MODES, UTCS, _collect, _cubes, _jupiter_series

pytestmark = pytest.mark.gpu


@pytest.fixture()
def L():
    from planetmapper_b200 import _lib

    return _lib


def _emission(L, frames, lons, lats):
    """(n_frames,) + grid EMISSION maps, from the launch the composite makes for that mask."""
    mask = L.mask_from_names(['PIXEL-X', 'PIXEL-Y', 'EMISSION'])
    maps = L.backplanes_map_batch(L.to_device(frames), L.to_device(np.asarray(lons) % 360), L.to_device(lats), mask)
    return maps[:, 2].cpu().numpy()


def _fold(mapped, emission, method, max_emission):
    """The composite rule on (n, nλ) + grid mapped values and (n,) + grid EMISSION, one epoch at a time in order."""
    shape = mapped.shape[1:]
    passes = np.ones(emission.shape, bool) if max_emission is None else emission <= max_emission
    if method == 'mean':
        total, count = np.zeros(shape), np.zeros(shape, np.int32)
        for f in range(len(mapped)):
            m = ~np.isnan(mapped[f]) & passes[f][None]
            total[m] = total[m] + mapped[f][m]
            count[m] += 1
        with np.errstate(invalid='ignore', divide='ignore'):
            return np.where(count > 0, total / count, np.nan), count
    value, key, tag = np.full(shape, np.nan), np.full(shape, np.nan), np.full(shape, -1, np.int32)
    for f in range(len(mapped)):
        e = np.broadcast_to(emission[f][None], shape)
        m = ~np.isnan(mapped[f]) & passes[f][None] & ~np.isnan(e) & ((tag < 0) | (e < key))
        value[m], key[m], tag[m] = mapped[f][m], e[m], f
    return value, tag


def _composite(S, *args, **kw):
    value, tag = S.composite_mapped_series(*args, **kw)
    assert value.is_cuda and tag.is_cuda
    return value.cpu().numpy(), tag.cpu().numpy()


def _series(nx=36, ny=28):
    import planetmapper_b200 as pm

    k = np.arange(len(UTCS))
    x0, y0, r0, rot = 17.0 + 0.4 * np.sin(k), 13.5 - 0.3 * k, 11.0 + 0.2 * k, 40.0 + 3.0 * k
    frames = _jupiter_series(UTCS, nx, ny, x0, y0, r0, rot)
    lons, lats, *_ = pm.BodyXY('Jupiter', UTCS[0], 'EARTH', nx=nx, ny=ny).generate_map_coordinates(degree_interval=7.5)
    return frames, lons, lats


def test_composite_equals_the_fold_of_the_mapped_series(L):
    from planetmapper_b200 import series as S

    nx, ny = 36, 28
    frames, lons, lats = _series(nx, ny)
    emission = _emission(L, frames, lons, lats)
    for nl in (1, 3, 5):
        cubes = _cubes(len(UTCS), nl, ny, nx, seed=nl)
        data = cubes[:, 0] if nl == 1 else cubes   # one image per epoch: 3-D input
        for mode in MODES:
            for prop in (True, False):
                mapped = _collect(S.iter_mapped_series(frames, data, nx, ny, lons, lats, interpolation=mode,
                                                       propagate_nan=prop, batch=3), len(UTCS))
                mapped = mapped.reshape((len(UTCS), nl) + lons.shape)
                for method in ('mean', 'min_emission'):
                    for cut in (None, 60.0):
                        got, tag = _composite(S, frames, data, nx, ny, lons, lats, interpolation=mode,
                                              propagate_nan=prop, method=method, max_emission=cut, batch=3)
                        want, want_tag = _fold(mapped, emission, method, cut)
                        if nl == 1:
                            want, want_tag = want[0], want_tag[0]
                        case = (nl, mode, prop, method, cut)
                        assert got.shape == want.shape and tag.dtype == np.int32, case
                        assert np.array_equal(got, want, equal_nan=True), case
                        assert np.array_equal(tag, want_tag), case
                        assert np.isfinite(got).sum() >= 100 * nl, case


def test_result_does_not_depend_on_the_batch():
    from planetmapper_b200 import series as S

    nx, ny = 36, 28
    frames, lons, lats = _series(nx, ny)
    cubes = _cubes(len(UTCS), 6, ny, nx, seed=11)
    for mode in ('nearest', 'linear', 'cubic', (2, 3)):
        for method, cut in (('mean', None), ('mean', 60.0), ('min_emission', None), ('min_emission', 60.0)):
            runs = [_composite(S, frames, cubes, nx, ny, lons, lats, interpolation=mode, method=method,
                               max_emission=cut, batch=b) for b in (1, 3, None)]
            for got, tag in runs[1:]:
                assert np.array_equal(got, runs[0][0], equal_nan=True), (mode, method, cut)
                assert np.array_equal(tag, runs[0][1]), (mode, method, cut)
            assert np.isfinite(runs[0][0]).sum() > 100 * 6


def test_mosaic_of_dithers():
    """One epoch repeated with four discs, each covering only part of the planet: EMISSION does not depend on the
    disc, so every dither that sees a cell ties there.  min_emission takes the lowest dither whose value is not NaN
    (cells outside a dither's image fall to the next one); mean averages exactly the covering dithers."""
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    nx, ny, nl = 24, 20, 3
    x0, y0 = np.array([3.0, 20.0, 3.0, 20.0]), np.array([3.0, 3.0, 16.0, 16.0])
    frames = _jupiter_series([UTCS[0]] * 4, nx, ny, x0, y0, 14.0, 30.0)
    lons, lats, *_ = pm.BodyXY('Jupiter', UTCS[0], 'EARTH', nx=nx, ny=ny).generate_map_coordinates(degree_interval=3)
    rng = np.random.default_rng(21)
    cubes = rng.normal(1.0, 0.3, (4, nl, ny, nx)) + np.arange(4)[:, None, None, None]
    cubes[rng.random(cubes.shape) < 0.02] = np.nan
    mapped = _collect(S.iter_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation='linear'), 4)
    covered = ~np.isnan(mapped)                          # (dither, plane) + grid
    assert (covered.sum(axis=0) >= 2).sum() > 50 * nl     # overlaps
    assert (covered.any(axis=0) & ~covered[0]).sum() > 50 * nl   # cells dither 0 does not see
    got, tag = _composite(S, frames, cubes, nx, ny, lons, lats, method='min_emission')
    first = np.where(covered.any(axis=0), np.argmax(covered, axis=0), -1)
    assert np.array_equal(tag, first)
    pick = np.take_along_axis(mapped, np.maximum(first, 0)[None], axis=0)[0]
    assert np.array_equal(got, np.where(first >= 0, pick, np.nan), equal_nan=True)
    assert set(np.unique(tag)) == {-1, 0, 1, 2, 3}
    got, count = _composite(S, frames, cubes, nx, ny, lons, lats, method='mean')
    assert np.array_equal(count, covered.sum(axis=0))
    total = np.zeros(mapped.shape[1:])
    for f in range(4):
        total = np.where(covered[f], total + np.nan_to_num(mapped[f]), total)
    with np.errstate(invalid='ignore'):
        assert np.array_equal(got, np.where(count > 0, total / count, np.nan), equal_nan=True)


def test_dense_map_cubic(L):
    """A 16 x 12 image onto the 1 deg grid (337 cells per image pixel): iter_mapped_series gathers a cube per
    epoch with the DMMA kernel, the composite with the scalar one, so the values agree to the last bits and the
    NaN masks and tags exactly; one image per epoch runs the scalar kernel in both and agrees bit for bit."""
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    nx, ny = 16, 12
    utcs = UTCS[:3] + UTCS[4:6] + UTCS[3:4]
    x0 = np.array([7.5, 7.2, 8.0, 7.6, 7.4, 7.0])
    frames = _jupiter_series(utcs, nx, ny, x0, 5.5, 5.0, 20.0)
    lons, lats, *_ = pm.BodyXY('Jupiter', utcs[0], 'EARTH', nx=nx, ny=ny).generate_map_coordinates(degree_interval=1)
    assert lons.size >= 20 * nx * ny
    emission = _emission(L, frames, lons, lats)
    for nl in (4, 5, 1):
        cubes = np.random.default_rng(nl).normal(1.0, 0.3, (len(utcs), nl, ny, nx))
        cubes[1, 0, 4, 5] = np.nan
        cubes[2, nl - 1] = np.nan
        data = cubes[:, 0] if nl == 1 else cubes
        for prop in (True, False):
            mapped = _collect(S.iter_mapped_series(frames, data, nx, ny, lons, lats, interpolation='cubic',
                                                   propagate_nan=prop, batch=4), len(utcs))
            mapped = mapped.reshape((len(utcs), nl) + lons.shape)
            for method, cut in (('mean', None), ('mean', 60.0), ('min_emission', None), ('min_emission', 75.0)):
                got, tag = _composite(S, frames, data, nx, ny, lons, lats, interpolation='cubic', propagate_nan=prop,
                                      method=method, max_emission=cut, batch=4)
                want, want_tag = _fold(mapped, emission, method, cut)
                case = (nl, prop, method, cut)
                if nl == 1:
                    assert np.array_equal(got, want[0], equal_nan=True), case
                    assert np.array_equal(tag, want_tag[0]), case
                    continue
                assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(tag, want_tag), case
                ok = np.isfinite(want)
                assert ok.sum() > 1000 * nl, case
                assert np.max(np.abs(got[ok] - want[ok])) <= 1e-12 * np.nanmax(np.abs(cubes)), case


def test_launches_per_batch_do_not_depend_on_its_epochs(L):
    from planetmapper_b200 import series as S

    nx, ny = 30, 26
    frames = _jupiter_series(UTCS, nx, ny, 14.5, 12.5, 10.0, 15.0)
    lo, la = np.meshgrid(np.arange(2.5, 360, 5.0)[::-1], np.arange(-87.5, 90, 5.0))
    for mode, nl, method, cut in (('nearest', 1, 'mean', None), ('nearest', 3, 'min_emission', None),
                                  ('linear', 1, 'mean', 60.0), ('cubic', 3, 'min_emission', 60.0),
                                  ((1, 2), 6, 'mean', None)):
        counts = []
        for n in (2, 7):
            cubes = _cubes(len(UTCS), nl, ny, nx, seed=3)[:n]
            before = L.launch_count()
            S.composite_mapped_series(frames[:n], cubes, nx, ny, lo, la, interpolation=mode, method=method,
                                      max_emission=cut, batch=n)
            counts.append(L.launch_count() - before)
        assert counts[0] == counts[1], (mode, nl, method, counts)
        if mode == 'nearest' and method == 'mean':
            assert counts[0] == 2   # the maps and the fold


def test_peak_memory_holds_no_per_epoch_output(L):
    """A cube composite allocates its accumulators, one batch's maps, staged cube and prepared operand: never the
    (batch, nλ) + grid output that iter_mapped_series fills and a fold would read back."""
    import torch

    from planetmapper_b200 import series as S

    n, nl, nx, ny = 7, 64, 32, 32
    frames = _jupiter_series(UTCS, nx, ny, 15.5, 15.5, 13.0, 10.0)
    lo, la = np.meshgrid(np.arange(0.5, 360, 1.0)[::-1], np.arange(-89.5, 90, 1.0))
    cubes = np.random.default_rng(2).normal(1.0, 0.3, (n, nl, ny, nx))
    lib = L.load_library()
    cells = lo.size
    for method, key_bytes in (('mean', 0), ('min_emission', 8)):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        value, tag = S.composite_mapped_series(frames, cubes, nx, ny, lo, la, interpolation='linear', method=method,
                                               max_emission=80.0, batch=n)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        planes = n * nl   # the batch's planes (stride nl: a multiple of 4)
        bound = (nl * cells * (8 + 4 + key_bytes)                 # accumulators
                 + n * 3 * cells * 8 + 2 * cells * 8 + n * 92 * 8  # maps, grid, frames
                 + planes * ny * nx * 8                            # staged cube
                 + lib.pm_spline_coef_bytes(planes, ny, nx) + lib.pm_spline_nanbits_bytes(planes, ny, nx)
                 + lib.pm_spline_planebits_bytes(planes) + lib.pm_spline_work_bytes(planes, ny, nx, L.INTERP_LINEAR)
                 + (4 << 20))                                      # allocator rounding
        output = n * nl * cells * 8
        assert peak <= bound < output, (method, peak, bound, output)
        assert np.isfinite(value.cpu().numpy()).sum() > 1000 * nl
        del value, tag
