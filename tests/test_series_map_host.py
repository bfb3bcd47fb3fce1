"""
Host side of the mapped time series (no GPU): the argument checks of pm_gather_grouped, the interpolation modes the
gather entry points accept, and the argument rules of series.iter_mapped_series, all before any device work.
"""
import ctypes

import numpy as np
import pytest

from planetmapper_b200 import _lib as L
from planetmapper_b200 import frame as F
from planetmapper_b200 import series as S

BAD, UNSUPPORTED = -1, -3


def test_grouped_gather_validates_arguments_before_device_work():
    lib = L.load_library()
    assert lib.pm_abi_version() == 10
    buf = np.zeros(64)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    g = lib.pm_gather_grouped  # src, nanbits, plane_bits, n_planes, ny, nx, n_maps, per_map, stride, xmaps, ymaps,
    #                            map_stride, n_cells, mode, flags, out, stream
    ok = [p, p, p, 12, 5, 6, 3, 4, 4, p, p, 10, 10, L.INTERP_CUBIC, L.FLAG_PROPAGATE_NAN, p, None]
    for i, v in ((3, -1), (4, 0), (5, 0), (6, -1), (6, 65536), (7, -1), (8, 3), (11, 9), (12, -1),
                 (3, 11),                       # the last group ends at plane 12
                 (4, 3), (5, 3),                # cubic needs ny, nx > 3
                 (11, 1 << 62)):                # map_stride * n_maps overflows
        args = list(ok)
        args[i] = v
        assert g(*args) == BAD, (i, v)
    for i in (0, 1, 2, 9, 10, 15):
        args = list(ok)
        args[i] = None
        assert g(*args) == BAD, i
    for mode in (-1, 4, L.INTERP_MIXED | 0x41, L.INTERP_MIXED | 0x10, 0x300 | 0x11):
        args = list(ok)
        args[13] = mode
        assert g(*args) == UNSUPPORTED, mode
    mixed = list(ok)
    mixed[13] = L.INTERP_MIXED | (1 << 4) | 3     # (1, 3): nx must exceed 3, ny only 1
    mixed[4], mixed[5] = 2, 3
    assert g(*mixed) == BAD
    # nearest reads the raw cube: no NaN words, any image size
    nearest = [p, None, None, 12, 1, 1, 3, 4, 4, p, p, 10, 10, L.INTERP_NEAREST, 0, None, None]
    assert g(*nearest) == BAD                      # out
    # empty input is valid with null pointers
    assert g(None, None, None, 0, 5, 6, 0, 4, 4, None, None, 0, 0, L.INTERP_CUBIC, 0, None, None) == 0
    assert g(None, None, None, 12, 5, 6, 3, 0, 4, None, None, 10, 10, L.INTERP_LINEAR, 0, None, None) == 0
    assert g(None, None, None, 12, 5, 6, 3, 4, 4, None, None, 10, 0, L.INTERP_NEAREST, 0, None, None) == 0


def test_gather_entry_points_agree_on_every_interpolation_mode():
    """pm_gather, pm_gather_grouped, pm_composite_grouped and pm_spline_prepare decode the interpolation mode alike:
    on a 1 x 1 image with no map cells a spline mode is refused for the image size, nearest is empty work (no spline
    to prepare) and every other code is unsupported; none of these calls reaches the device."""
    lib = L.load_library()
    buf = np.zeros(64)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    splines = {L.INTERP_LINEAR, L.INTERP_QUADRATIC, L.INTERP_CUBIC}
    splines |= {L.INTERP_MIXED | (ky << 4) | kx for ky in (1, 2, 3) for kx in (1, 2, 3)}
    for mode in range(-2, 0x400):
        want = BAD if mode in splines else 0 if mode == L.INTERP_NEAREST else UNSUPPORTED
        assert lib.pm_gather(p, p, p, 1, 1, 1, 0, 1, p, p, 0, 0, mode, 0, p, None) == want, mode
        assert lib.pm_gather_grouped(p, p, p, 1, 1, 1, 1, 1, 1, p, p, 0, 0, mode, 0, p, None) == want, mode
        assert lib.pm_composite_grouped(p, p, p, 1, 1, 1, 1, 1, 1, p, 2, 0, 0, mode, 0, 0, float('inf'), 0, 1, 1, p,
                                        None, p, None) == want, mode
        want = UNSUPPORTED if mode == L.INTERP_NEAREST else want
        assert lib.pm_spline_prepare(p, 1, 1, 1, mode, p, p, p, p, None) == want, mode


def _args(n=3, nl=None, ny=8, nx=9):
    frames = np.zeros((n, F.PMFRAME_NDOUBLES))
    cubes = np.zeros((n, ny, nx) if nl is None else (n, nl, ny, nx))
    lons, lats = np.meshgrid(np.arange(5.0), np.arange(4.0))
    return frames, cubes, nx, ny, lons, lats


def test_iter_mapped_series_argument_rules_need_no_device(monkeypatch):
    def no_device():
        raise AssertionError('touched the device')

    monkeypatch.setattr(L, '_torch', no_device)
    monkeypatch.setattr(L, 'to_device', lambda *a, **k: no_device())
    frames, cubes, nx, ny, lons, lats = _args()
    for kw in (dict(interpolation='smooth'), dict(spline_smoothing=0.5), dict(interpolation='cubic', spline_smoothing=0.5),
               dict(interpolation=4), dict(interpolation=(4, 1)), dict(interpolation=5)):
        with pytest.raises(NotImplementedError):
            S.iter_mapped_series(frames, cubes, nx, ny, lons, lats, **kw)
    with pytest.raises(ValueError, match='Unknown interpolation'):
        S.iter_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation='bicubic')
    bad = [
        (np.zeros((3, 91)), cubes, nx, ny, lons, lats),              # frames
        (frames, np.zeros((2, ny, nx)), nx, ny, lons, lats),         # one cube per frame
        (frames, np.zeros((3, ny, nx + 1)), nx, ny, lons, lats),     # image size
        (frames, np.zeros((3, 2, ny + 1, nx)), nx, ny, lons, lats),
        (frames, np.zeros((3, 0, ny, nx)), nx, ny, lons, lats),      # no planes
        (frames, np.zeros((3, 1, 1, ny, nx)), nx, ny, lons, lats),   # 5-D
        (frames, np.zeros((ny, nx)), nx, ny, lons, lats),
        (frames, cubes, nx, ny, lons, lats[:2]),                    # grid
        (frames, cubes, nx, ny, lons[:0], lats[:0]),
    ]
    for args in bad:
        with pytest.raises(ValueError):
            S.iter_mapped_series(*args)
    with pytest.raises(ValueError):
        S.iter_mapped_series(*_args(), batch=0)


def test_series_stride_puts_spline_cubes_on_plane_quads():
    assert [S._series_stride(n, L.INTERP_CUBIC) for n in (1, 2, 3, 4, 5, 8, 9)] == [1, 4, 4, 4, 8, 8, 12]
    assert [S._series_stride(n, L.INTERP_MIXED | 0x13) for n in (1, 3)] == [1, 4]
    assert [S._series_stride(n, L.INTERP_NEAREST) for n in (1, 3, 5)] == [1, 3, 5]
