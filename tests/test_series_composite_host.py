"""
Host side of the composite of a mapped series (no GPU): the argument checks of pm_composite_grouped and the argument
rules of series.composite_mapped_series, both before any device work.
"""
import ctypes
import math

import numpy as np
import pytest

from planetmapper_b200 import _lib as L
from planetmapper_b200 import frame as F
from planetmapper_b200 import series as S

BAD, UNSUPPORTED = -1, -3
MEAN, MIN_EMISSION = 0, 1
INF = math.inf


def test_composite_validates_arguments_before_device_work():
    lib = L.load_library()
    assert lib.pm_abi_version() == 10
    buf = np.zeros(64)
    p = buf.ctypes.data_as(ctypes.c_void_p)
    c = lib.pm_composite_grouped
    # src, nanbits, plane_bits, n_planes, ny, nx, n_maps, per_map, stride, maps, n_map_planes, map_stride, n_cells,
    # mode, flags, method, max_emission, epoch_begin, first, last, value, key, tag, stream
    ok = [p, p, p, 12, 5, 6, 3, 4, 4, p, 3, 30, 10, L.INTERP_CUBIC, L.FLAG_PROPAGATE_NAN, MIN_EMISSION, 60.0, 0, 1, 0,
          p, p, p, None]
    for i, v in ((3, -1), (4, 0), (5, 0), (6, -1), (6, 65536), (7, -1), (8, 3), (12, -1),
                 (3, 11),                        # the last epoch's planes end at plane 12
                 (4, 3), (5, 3),                 # cubic needs ny, nx > 3
                 (10, 1), (10, 4), (10, 2),      # map planes: x, y, EMISSION (min_emission needs EMISSION)
                 (11, 29),                       # an epoch's three map planes of 10 cells
                 (11, 1 << 62),                  # map_stride * n_maps overflows
                 (14, 4), (14, 1),               # flags: only propagate_nan
                 (16, math.nan),                 # the EMISSION cut
                 (17, -1), (17, 2 ** 31 - 3),    # epoch_begin (+ n_maps must fit an int32 tag)
                 (18, 2), (19, -1)):             # first / last are 0 or 1
        args = list(ok)
        args[i] = v
        assert c(*args) == BAD, (i, v)
    for i in (0, 1, 2, 9, 20, 21, 22):
        args = list(ok)
        args[i] = None
        assert c(*args) == BAD, i
    for i, v in ((13, -1), (13, 4), (13, L.INTERP_MIXED | 0x41), (13, L.INTERP_MIXED | 0x10), (13, 0x300 | 0x11),
                 (15, -1), (15, 2)):
        args = list(ok)
        args[i] = v
        assert c(*args) == UNSUPPORTED, (i, v)
    # a mean without EMISSION: no cut, and no key
    mean = list(ok)
    mean[10], mean[15], mean[16], mean[21] = 2, MEAN, INF, None
    for i, v in ((16, 60.0), (16, 180.0), (15, MIN_EMISSION)):
        args = list(mean)
        args[i] = v
        assert c(*args) == BAD, (i, v)
    # nearest reads the raw cube: no NaN words, any image size
    nearest = list(mean)
    nearest[1], nearest[2], nearest[4], nearest[5], nearest[13], nearest[14] = None, None, 1, 1, L.INTERP_NEAREST, 0
    for i in (0, 9, 20, 22):
        args = list(nearest)
        args[i] = None
        assert c(*args) == BAD, i
    # empty input is valid with null pointers
    assert c(None, None, None, 0, 5, 6, 0, 4, 4, None, 3, 0, 0, L.INTERP_CUBIC, 0, MIN_EMISSION, 60.0, 0, 1, 1,
             None, None, None, None) == 0
    assert c(None, None, None, 12, 5, 6, 3, 0, 4, None, 2, 20, 10, L.INTERP_LINEAR, 0, MEAN, INF, 0, 1, 1,
             None, None, None, None) == 0
    assert c(None, None, None, 12, 5, 6, 3, 4, 4, None, 3, 0, 0, L.INTERP_NEAREST, 0, MEAN, 0.0, 0, 0, 0,
             None, None, None, None) == 0


def _args(n=3, nl=None, ny=8, nx=9):
    frames = np.zeros((n, F.PMFRAME_NDOUBLES))
    cubes = np.zeros((n, ny, nx) if nl is None else (n, nl, ny, nx))
    lons, lats = np.meshgrid(np.arange(5.0), np.arange(4.0))
    return frames, cubes, nx, ny, lons, lats


def test_composite_argument_rules_need_no_device(monkeypatch):
    def no_device():
        raise AssertionError('touched the device')

    monkeypatch.setattr(L, '_torch', no_device)
    monkeypatch.setattr(L, 'to_device', lambda *a, **k: no_device())
    frames, cubes, nx, ny, lons, lats = _args()
    # iter_mapped_series' refusals, with its exception types
    for kw in (dict(interpolation='smooth'), dict(spline_smoothing=0.5), dict(interpolation='cubic', spline_smoothing=0.5),
               dict(interpolation=4), dict(interpolation=(4, 1)), dict(interpolation=5)):
        with pytest.raises(NotImplementedError):
            S.composite_mapped_series(frames, cubes, nx, ny, lons, lats, **kw)
    with pytest.raises(ValueError, match='Unknown interpolation'):
        S.composite_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation='bicubic')
    bad = [
        (np.zeros((3, 91)), cubes, nx, ny, lons, lats),              # frames
        (frames, np.zeros((2, ny, nx)), nx, ny, lons, lats),         # one cube per frame
        (frames, np.zeros((3, ny, nx + 1)), nx, ny, lons, lats),     # image size
        (frames, np.zeros((3, 0, ny, nx)), nx, ny, lons, lats),      # no planes
        (frames, np.zeros((3, 1, 1, ny, nx)), nx, ny, lons, lats),   # 5-D
        (frames, cubes, nx, ny, lons, lats[:2]),                    # grid
        (frames, cubes, nx, ny, lons[:0], lats[:0]),
        (frames[:0], cubes[:0], nx, ny, lons, lats),                # no epoch to composite
    ]
    for args in bad:
        with pytest.raises(ValueError):
            S.composite_mapped_series(*args)
    for kw in (dict(batch=0), dict(method='median'), dict(method='MEAN'), dict(max_emission=math.nan),
               dict(max_emission=-1.0), dict(max_emission=180.5), dict(max_emission=INF),
               dict(method='min_emission', max_emission=-0.1)):
        with pytest.raises(ValueError):
            S.composite_mapped_series(*_args(), **kw)
