"""
Host side of the mapped time series (no GPU): the argument checks of pm_gather_grouped and the argument rules of
series.iter_mapped_series, both before any device work.
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
