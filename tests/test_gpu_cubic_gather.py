"""
The dense-map cubic gather (gather_cubic_mma_kernel) on every path it takes, driven on purpose with
constructed x / y maps and checked against three references that share no code with it:

- scipy: oracle/map_img_oracle.map_cube_fast, the real RectBivariateSpline(s=0).ev after the reference's NaN
  repair: identical NaN masks and at most 1e-10 relative difference;
- an exact polynomial: a not-a-knot cubic reproduces p(u, v) = sum c_ij u^i v^j (i, j <= 3) exactly, so the
  map is p at the clamped cell coordinates, evaluated in long double: at most 1e-11 of max |p| over the image;
- the one-cell-per-thread kernel gather_spline_kernel<4, 4>, bit for bit: the same cells launched in flat
  chunks below the launcher's density rule.  For every cell the DMMA kernel adds the same nonzero products in
  the same order (row j outer, column inner) and its masked products add exact zeros.

The kernel picks its path per warp from data: 1-D cell order or 4 x 8 cell blocks (narrow maps), a pipeline
for one to four distinct 4 x 4 footprints in the warp, a general path for more, NaN streaming for a warp with
no valid cell.  A single real-geometry map does not reliably reach the rare ones, so each warp's 32 cells are
filled from a pattern (warp_lanes / build_map below).  test_constructed_maps_reach_every_path checks, without
a GPU, that the maps contain every pattern and that each launch selects the kernel it is meant to test.
"""
import functools
import math
import zlib
from collections import namedtuple

import numpy as np
import pytest

from conftest import GOLDEN_DISC
from test_gpu_parity import _cube

MMA_KERNEL = 'gather_cubic_mma_kernel'
SCALAR_KERNEL = 'gather_spline_kernel'
DENSITY = 20            # map cells per image pixel from which the DMMA kernel runs (gather_kernels.cu:854)
SCIPY_BAR = 1e-10       # |got - scipy| / max(|scipy|, 1)
POLY_BAR = 1e-11        # |got - p| / max |p| over the image


def select_kernel(n_cells, nx, ny, cells_per_row):
    """The kernel launch_gather runs for a cubic gather (gather_kernels.cu:854-869): 'dense-1d' (DMMA, 32
    consecutive cells per warp), 'dense-2d' (DMMA, 4 map rows x 8 columns per warp) or 'scalar'
    (gather_spline_kernel<4, 4>, one cell per thread).  cells_per_row is the map's last dimension, 0 for a
    flat map (_lib.gather)."""
    if not (n_cells >= DENSITY * nx * ny and nx < 16384 and ny < 16384):
        return 'scalar'
    rows_ok = 0 < cells_per_row < 64 and cells_per_row < n_cells and n_cells % cells_per_row == 0
    return 'dense-2d' if rows_ok else 'dense-1d'


def warp_lanes(shape):
    """Warp and lane of every cell (row-major) of a map of `shape`, as gather_cubic_mma_kernel assigns them
    (gather_kernels.cu:339-358): lane = 8 * tile + column.  A 2-D map whose rows are shorter than 64 cells is
    cut into blocks of 4 rows x 8 columns (tile = row of the block, blocks numbered row-group major); any
    other map into runs of 32 consecutive cells (tile = cells 8 i .. 8 i + 7)."""
    n = math.prod(shape)
    row_len = shape[-1] if len(shape) >= 2 else 0
    cell = np.arange(n)
    if 0 < row_len < 64 and row_len < n and n % row_len == 0:
        r, c = np.divmod(cell, row_len)
        warp = (r // 4) * ((row_len + 7) // 8) + c // 8
        lane = 8 * (r % 4) + c % 8
    else:
        warp, lane = np.divmod(cell, 32)
    return warp, lane


def footprint_origin(v, n):
    """First coefficient index of the cubic footprint along an axis of n samples (bspline_weights,
    gather_kernels.cu:45-72): clamp(floor(clamp(v, 0, n-1)) - 1, 0, n - 4)."""
    return np.clip(np.floor(np.clip(v, 0, n - 1)) - 1, 0, n - 4).astype(np.int64)


# ---- constructed maps -------------------------------------------------------------------------------------
PATTERNS = ('nf1', 'nf2x', 'nf2y', 'nf3x', 'nf3y', 'nf4', 'scatter', 'edge', 'nan')
_WEIGHTS = dict(nf1=6, nf2x=3, nf2y=3, nf3x=2, nf3y=2, nf4=3, scatter=3, edge=3, nan=2)


def patterns_for(nx, ny):
    """The patterns an image has room for: nf<k><axis> needs k footprint origins along that axis (n - 3 of
    them for n samples), nf4 a 2 x 2 corner of them, scatter at least five."""
    mx, my = nx - 3, ny - 3
    ok = dict(nf1=True, nf2x=mx >= 2, nf2y=my >= 2, nf3x=mx >= 3, nf3y=my >= 3, nf4=mx >= 2 and my >= 2,
              scatter=mx * my >= 5, edge=True, nan=True)
    return [p for p in PATTERNS if ok[p]]


def _pick(rng, m):
    """An origin in [0, m), the first or last one a third of the time (footprints at the frame's edges cover
    two image pixels along that axis, and the last ones carry the largest packed pixel indices)."""
    if rng.random() < 1 / 3:
        return 0 if rng.random() < 0.5 else m - 1
    return int(rng.integers(m))


def _axis_sample(rng, o, n, size):
    """Coordinates in [0, n-1] whose footprint origin along the axis is o; a fifth of them on integers, where
    the NaN test reads one pixel instead of two."""
    lo = 0.0 if o == 0 else o + 1.0
    hi = n - 1.0 if o == n - 4 else o + 2.0
    v = rng.uniform(lo, hi, size)
    ints = np.arange(math.ceil(lo), math.floor(hi) + 1, dtype=float)
    if o < n - 4:
        ints = ints[ints < hi]
    on = rng.random(size) < 0.2
    v[on] = rng.choice(ints, int(on.sum()))
    return v


def edge_values(n):
    """Coordinates at and around the edges of an axis of n samples: the edges themselves, just inside and just
    outside them (1e-12, or two units in the last place where that is coarser), and far outside."""
    eps = max(1e-12, 2 * float(np.spacing(float(n - 1))))
    return np.array([0.0, n - 1.0, 1e-12, -1e-12, n - 1 - eps, n - 1 + eps, -5.0, n + 3.0, 1.0, n - 2.0])


def make_pattern(rng, kind, nx, ny):
    """x, y of the 32 lanes of one warp."""
    if kind == 'nan':
        return np.full(32, np.nan), np.full(32, np.nan)
    if kind == 'edge':
        xy = []
        for n in (nx, ny):
            v = rng.uniform(0, n - 1, 32)
            e = rng.random(32) < 0.7
            v[e] = rng.choice(edge_values(n), int(e.sum()))
            xy.append(v)
        return xy[0], xy[1]
    mx, my = nx - 3, ny - 3
    if kind == 'scatter':
        k = int(rng.integers(5, min(32, mx * my) + 1))
        flat = rng.choice(mx * my, k, replace=False)
        fps = [(int(f % mx), int(f // mx)) for f in flat]
    else:
        ax, ay = dict(nf1=(1, 1), nf2x=(2, 1), nf2y=(1, 2), nf3x=(3, 1), nf3y=(1, 3), nf4=(2, 2))[kind]
        ox, oy = _pick(rng, mx - ax + 1), _pick(rng, my - ay + 1)
        fps = [(ox + i, oy + j) for j in range(ay) for i in range(ax)]
    k = len(fps)
    style = 'random' if kind == 'scatter' else rng.choice(['random', 'runs', 'tiles'])
    which = rng.integers(k, size=32)
    which[rng.permutation(32)[:k]] = np.arange(k)           # every footprint is read by some lane
    if style == 'runs':                                      # contiguous runs, as along a real map row
        which = np.sort(which)
    elif style == 'tiles' and k > 1:                         # tiles 0 and 1 read one footprint each, 2 and 3 mix
        which[0:8], which[8:16] = 0, 1
        which[16:16 + k] = np.arange(k)
    x, y = np.empty(32), np.empty(32)
    for f, (ox, oy) in enumerate(fps):
        m = which == f
        x[m] = _axis_sample(rng, ox, nx, int(m.sum()))
        y[m] = _axis_sample(rng, oy, ny, int(m.sum()))
    if rng.random() < 0.25:                                  # a few cells off the disc
        off = rng.permutation(32)[:int(rng.integers(1, 9))]
        x[off] = y[off] = np.nan
    return x, y


Case = namedtuple('Case', 'name nx ny shape cubes kernel')
_C600 = (('c600', ((0, 600), (4, 5), (28, 9), (4, 596))),)
_SMALL = (('c37', ((0, 37), (4, 5), (28, 9))), ('c3', ((0, 3),)), ('c1', ((0, 1),)))
_C3 = (('c3', ((0, 3),)),)
CASES = [
    # flat maps: even and a multiple of 32, odd, even with a ragged last warp
    Case('12x9-flat-8640', 12, 9, (8640,), _C600, 'dense-1d'),
    Case('12x9-flat-8641', 12, 9, (8641,), _C600, 'dense-1d'),
    Case('12x9-flat-8650', 12, 9, (8650,), _C600, 'dense-1d'),
    # narrow maps: 4 x 8 cell blocks, a row count that is not a multiple of 4, ragged column tiles
    Case('12x9-rows-8', 12, 9, (1083, 8), _C600, 'dense-2d'),
    Case('12x9-rows-13', 12, 9, (667, 13), _C600, 'dense-2d'),
    Case('12x9-rows-40', 12, 9, (217, 40), _C600, 'dense-2d'),
    Case('12x9-rows-63', 12, 9, (138, 63), _C600, 'dense-2d'),
    # the smallest cubic image
    Case('4x5-flat-1601', 4, 5, (1601,), _SMALL, 'dense-1d'),
    Case('4x5-rows-13', 4, 5, (123, 13), _SMALL, 'dense-2d'),
    # the 14-bit limits of the packed NaN-test pixels (nbp), and one column past them
    Case('16383x4-flat', 16383, 4, (1310641,), _C3, 'dense-1d'),
    Case('4x16383-rows-40', 4, 16383, (32767, 40), _C3, 'dense-2d'),
    Case('16384x4-flat', 16384, 4, (1310721,), _C3, 'scalar'),
]
CASES_BY_NAME = {c.name: c for c in CASES}


MAX_PATTERN_WARPS = 2048   # on the 1.3 M-cell maps; the other warps read one random footprint each


@functools.lru_cache(maxsize=None)
def build_map(name):
    """x, y maps of a case, filled warp by warp from random patterns, and the pattern of every warp.  On maps
    of more than MAX_PATTERN_WARPS warps, that many random warps (the last one included) get a pattern and the
    others ('bulk') one footprint each, drawn vectorised."""
    c = CASES_BY_NAME[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    warp, lane = warp_lanes(c.shape)
    n_warps = int(warp.max()) + 1
    X, Y = np.empty((n_warps, 32)), np.empty((n_warps, 32))
    for V, n in ((X, c.nx), (Y, c.ny)):
        o = rng.integers(n - 3, size=(n_warps, 1))
        lo = np.where(o == 0, 0.0, o + 1.0)
        hi = np.where(o == n - 4, n - 1.0, o + 2.0)
        V[:] = lo + (hi - lo) * rng.random((n_warps, 32))
    pattern = np.full(n_warps, 'bulk', dtype='<U8')
    chosen = np.arange(n_warps)
    if n_warps > MAX_PATTERN_WARPS:
        chosen = np.append(rng.choice(n_warps - 1, MAX_PATTERN_WARPS - 1, replace=False), n_warps - 1)
    kinds = patterns_for(c.nx, c.ny)
    p = np.array([_WEIGHTS[k] for k in kinds], dtype=float)
    for w, k in zip(chosen, rng.choice(len(kinds), chosen.size, p=p / p.sum())):
        X[w], Y[w] = make_pattern(rng, kinds[k], c.nx, c.ny)
        pattern[w] = kinds[k]
    return X[warp, lane].reshape(c.shape), Y[warp, lane].reshape(c.shape), pattern


def lane_matrix(name, values, fill=np.nan):
    """Per-cell values of a case as (warps, 32 lanes); lanes without a cell (ragged warps) hold `fill`."""
    warp, lane = warp_lanes(CASES_BY_NAME[name].shape)
    m = np.full((int(warp.max()) + 1, 32), fill, dtype=np.asarray(values).dtype)
    m[warp, lane] = np.asarray(values).reshape(-1)
    return m


def valid_cells(x, y, nx, ny, propagate):
    """Cells the kernel evaluates: x not NaN and, with propagate_nan, inside the frame."""
    v = ~np.isnan(x)
    if propagate:
        with np.errstate(invalid='ignore'):
            v &= (x >= 0) & (y >= 0) & (x <= nx - 1) & (y <= ny - 1)
    return v


def distinct(keys):
    """Number of distinct keys per row of a 2-D integer array (keys < 0 ignored)."""
    s = np.sort(keys, axis=1)
    new = np.ones(s.shape, dtype=bool)
    new[:, 1:] = s[:, 1:] != s[:, :-1]
    return (new & (s >= 0)).sum(axis=1)


def lane_origins(name, propagate):
    """(warps, 32) footprint origins along x and y of the cells the kernel evaluates, -1 elsewhere."""
    c = CASES_BY_NAME[name]
    x, y, _ = build_map(name)
    X, Y = lane_matrix(name, x), lane_matrix(name, y)
    v = valid_cells(X, Y, c.nx, c.ny, propagate)
    ox = np.where(v, footprint_origin(np.nan_to_num(X), c.nx), -1)
    oy = np.where(v, footprint_origin(np.nan_to_num(Y), c.ny), -1)
    return ox, oy


def warp_paths(name, propagate):
    """Per warp: the number of distinct footprints among its valid cells (the kernel's org0..org3 / `simple`)
    and the path that number selects: 'none' (NaN streaming), 'nf1' .. 'nf4' (pipeline), 'general'."""
    ox, oy = lane_origins(name, propagate)
    nf = distinct(np.where(ox >= 0, oy * CASES_BY_NAME[name].nx + ox, -1))
    path = np.where(nf == 0, 'none', np.where(nf <= 4, np.char.add('nf', nf.astype(str)), 'general'))
    return nf, path


# ---- cubes ------------------------------------------------------------------------------------------------
POLY_PLANES = {'c600': list(range(33, 37)) + list(range(64, 96)) + list(range(596, 600)),
               'c37': list(range(8, 16)) + list(range(33, 37)), 'c3': [0, 2], 'c1': [0]}


def poly_eval(c, x, y, nx, ny):
    """p(u, v) = sum c[i, j] u^i v^j at u = x / (nx - 1), v = y / (ny - 1), in long double."""
    u = np.asarray(x, dtype=np.longdouble) / (nx - 1)
    v = np.asarray(y, dtype=np.longdouble) / (ny - 1)
    out = np.zeros(np.broadcast(u, v).shape, dtype=np.longdouble)
    for i in range(4):
        for j in range(4):
            out += np.longdouble(c[i, j]) * u ** i * v ** j
    return out


@functools.lru_cache(maxsize=None)
def make_cube(kind, nx, ny):
    """(cube, {plane: polynomial coefficients}).  c600 / c37: the NaN layouts of test_gpu_parity._cube in
    planes 0-7 (isolated, scattered, block and row NaN, an all-NaN plane, inf pixels, an all-inf plane),
    all-NaN planes 31 and 32, a few NaN pixels per other plane, NaN-free polynomial planes (c600: all of
    planes 64-95, a 32-plane word without NaN).  c3: polynomial, noise with NaN and an inf pixel, polynomial.
    c1: one polynomial plane (a cube without NaN)."""
    rng = np.random.default_rng(zlib.crc32(f'{kind} {nx} {ny}'.encode()))
    nl = int(kind[1:])
    if nl >= 8:
        cube = _cube(rng, nl, ny, nx)
        cube[8:][rng.random((nl - 8, ny, nx)) < max(0.01, 1.5 / (nx * ny))] = np.nan
        cube[31:33] = np.nan
    else:
        cube = rng.normal(1.0, 0.1, (nl, ny, nx))
        if nl == 3:
            cube[1][rng.random((ny, nx)) < 0.02] = np.nan
            cube[1, ny // 2, 1] = np.nan
            cube[1, 0, nx // 2] = np.inf
    yy, xx = np.mgrid[0:ny, 0:nx]
    poly = {}
    for l in POLY_PLANES[kind]:
        poly[l] = rng.normal(size=(4, 4))
        cube[l] = poly_eval(poly[l], xx, yy, nx, ny).astype(np.float64)
    return cube, poly


def scipy_cells(name):
    """Cells compared with scipy: all of them, except on the 1.3 M-cell maps, where FITPACK's knot search is
    linear in the coordinate (~5 us per cell along a 16383-sample axis): there the patterned warps and 256
    random bulk warps."""
    c = CASES_BY_NAME[name]
    warp, _ = warp_lanes(c.shape)
    _, _, pattern = build_map(name)
    keep = pattern != 'bulk'
    if not keep.all():
        rng = np.random.default_rng(1)
        keep[rng.choice(np.flatnonzero(~keep), 256, replace=False)] = True
    return keep[warp]


# ---- premise (no GPU) -------------------------------------------------------------------------------------
def test_constructed_maps_reach_every_path():
    """The maps drive every path of the kernel they are meant to, and each launch of the GPU tests selects the
    kernel it is meant to test.  A move of the launcher's density rule or cell layout shows here first."""
    flat = [c for c in CASES if len(c.shape) == 1 and c.kernel != 'scalar']
    assert {c.shape[0] % 2 for c in flat} == {0, 1} and any(c.shape[0] % 32 for c in flat if c.shape[0] % 2 == 0)
    rows = [c for c in CASES if len(c.shape) == 2]
    assert {8, 13, 40, 63} <= {c.shape[1] for c in rows} and all(c.shape[0] % 4 for c in rows)
    assert {(16383, 4), (4, 16383), (16384, 4), (4, 5), (12, 9)} <= {(c.nx, c.ny) for c in CASES}
    assert select_kernel(40 * 40, GOLDEN_DISC['nx'], GOLDEN_DISC['ny'], 40) == 'dense-2d'   # the map_img test

    seen_paths = set()
    for c in CASES:
        n = math.prod(c.shape)
        assert select_kernel(n, c.nx, c.ny, c.shape[-1] if len(c.shape) == 2 else 0) == c.kernel, c.name
        chunk = DENSITY * c.nx * c.ny - 1                  # the bit-exact reference: flat chunks, scalar kernel
        assert select_kernel(chunk, c.nx, c.ny, 0) == 'scalar' and chunk < n, c.name
        x, y, pattern = build_map(c.name)
        assert set(pattern) - {'bulk'} == set(patterns_for(c.nx, c.ny)), c.name
        for v, m in ((x, c.nx), (y, c.ny)):                # every edge value and edge pixel on both axes
            assert np.isin(edge_values(m), v).all(), c.name
            assert np.isin(np.arange(m, dtype=float)[[0, 1, -2, -1]], v).all(), c.name
        X, Y = lane_matrix(c.name, x), lane_matrix(c.name, y)
        present = lane_matrix(c.name, np.ones(n, dtype=bool), False)
        nan = np.isnan(X) & present
        assert (nan.any(1) & (nan.sum(1) < present.sum(1))).sum() >= 5, c.name   # warps with some cells NaN
        mx, my = c.nx - 3, c.ny - 3                        # footprint origins per axis
        for prop in (True, False):
            nf, path = warp_paths(c.name, prop)
            counts = {p: int((path == p).sum()) for p in ('none', 'nf1', 'nf2', 'nf3', 'nf4', 'general')}
            possible = dict(none=True, nf1=True, nf2=max(mx, my) >= 2, nf3=max(mx, my) >= 3,
                            nf4=mx >= 2 and my >= 2, general=mx * my >= 5)
            assert all(counts[p] >= 3 for p in counts if possible[p]), (c.name, prop, counts)
            seen_paths |= {p for p in counts if counts[p]}
            ox, oy = lane_origins(c.name, prop)
            org = np.where(ox >= 0, oy * c.nx + ox, -1)
            # two and three footprints along one axis: they share a row (along x) or a column (along y) of origins
            along_x, along_y = distinct(oy) == 1, distinct(ox) == 1
            for k in (2, 3):
                assert mx < k or ((nf == k) & along_x).sum() >= 3, (c.name, prop, k)
                assert my < k or ((nf == k) & along_y).sum() >= 3, (c.name, prop, k)
            # two to four footprints, one tile reading one footprint (`tiles` bit 16 + i) and another mixing them
            if mx * my >= 2:
                per_tile = distinct(org.reshape(-1, 8)).reshape(-1, 4)
                mixed = (per_tile == 1).any(1) & (per_tile >= 2).any(1) & (nf >= 2) & (nf <= 4)
                assert mixed.sum() >= 3, (c.name, prop)
            # one footprint whose cells test different pixels for NaN (x0 | y0 | x1 > x0 | y1 > y0 of nbp)
            Xs, Ys = np.nan_to_num(X), np.nan_to_num(Y)
            x0, y0 = np.maximum(np.floor(Xs), 0), np.maximum(np.floor(Ys), 0)
            dx, dy = np.minimum(np.ceil(Xs), c.nx - 1) > x0, np.minimum(np.ceil(Ys), c.ny - 1) > y0
            nb = np.where(ox >= 0, ((y0 * c.nx + x0) * 4 + 2 * dy + dx).astype(np.int64), -1)
            assert ((nf == 1) & (distinct(nb) > 1)).sum() >= 3, (c.name, prop)
            # cells outside the frame: evaluated clamped (propagate_nan=False) or NaN (True)
            with np.errstate(invalid='ignore'):
                outside = present & ~np.isnan(X) & ((X < 0) | (Y < 0) | (X > c.nx - 1) | (Y > c.ny - 1))
            assert outside.sum() >= 100 and ((ox[outside] >= 0) == (not prop)).all(), c.name
    assert seen_paths == {'none', 'nf1', 'nf2', 'nf3', 'nf4', 'general'}

    for kind, ranges in _C600 + _SMALL:
        cube, poly = make_cube(kind, 12, 9)
        nl = cube.shape[0]
        assert all(b % 4 == 0 and b + n <= nl for b, n in ranges)
        assert all(np.isfinite(cube[l]).all() for l in poly)
    cube, poly = make_cube('c600', 12, 9)
    assert np.isnan(cube[31]).all() and np.isnan(cube[32]).all() and np.isinf(cube[5]).any()
    assert not np.isnan(cube[64:96]).any() and np.isnan(cube[96:128]).any()   # one NaN-free 32-plane word
    assert (4, 596) in _C600[0][1] and 596 + 4 > 512                           # lead = 4 and two plane groups


# ---- GPU ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def L():
    import torch

    from planetmapper_b200 import _lib

    assert torch.cuda.is_available()
    _lib.load_library()
    return _lib


def scalar_launch(L, spline, xd, yd, nx, ny, begin, count, propagate):
    """The same cells as flat chunks below the density rule: gather_spline_kernel<4, 4>."""
    import torch

    xf, yf = xd.reshape(-1), yd.reshape(-1)
    chunk = DENSITY * nx * ny - 1
    parts = [L.gather(spline, xf[s:s + chunk], yf[s:s + chunk], L.INTERP_CUBIC, plane_begin=begin,
                      plane_count=count, propagate_nan=propagate) for s in range(0, xf.numel(), chunk)]
    return torch.cat(parts, dim=1)


def _rel_vs_scipy(got, ref, label):
    mism = np.isnan(got) != np.isnan(ref)
    assert not mism.any(), f'{label}: {int(mism.sum())} NaN-mask differences from scipy'
    rel = np.zeros(ref.shape)
    fin = np.isfinite(ref)
    rel[fin] = np.abs(got[fin] - ref[fin]) / np.maximum(np.abs(ref[fin]), 1.0)
    assert rel.max(initial=0.0) <= SCIPY_BAR, f'{label}: rel {rel.max():.3e} vs scipy'
    return rel


def _rel_vs_poly(got, want, scale, label):
    """got (cells,), want (cells,) long double with NaN where the cell must be NaN."""
    mism = np.isnan(got) != np.isnan(want)
    assert not mism.any(), f'{label}: {int(mism.sum())} NaN-mask differences from the polynomial'
    fin = ~np.isnan(want)
    rel = np.zeros(got.shape)
    rel[fin] = np.abs(got[fin].astype(np.longdouble) - want[fin]) / scale
    assert rel.max(initial=0.0) <= POLY_BAR, f'{label}: rel {rel.max():.3e} of max |p| vs the polynomial'
    return rel


@pytest.mark.gpu
@pytest.mark.timeout(300, method='thread')
@pytest.mark.parametrize('name', [c.name for c in CASES])
def test_cubic_gather_vs_scipy_polynomial_and_scalar_kernel(L, name):
    """Every plane range and both propagate_nan values against all three references; every disagreement is
    reported, not only the first.  The worst relative errors per kernel path go to the parity report."""
    import torch

    from helpers import write_parity_report
    from oracle import map_img_oracle as MO

    c = CASES_BY_NAME[name]
    x, y, _ = build_map(name)
    xd, yd = L.to_device(x), L.to_device(y)
    xf, yf = x.reshape(-1), y.reshape(-1)
    sub = scipy_cells(name)
    report = {'kernel': c.kernel, 'cells': int(xf.size), 'cells_vs_scipy': int(sub.sum()),
              'bit_equal_to_scalar_kernel': 'compared' if c.kernel != 'scalar' else 'is the scalar kernel'}
    failures = []

    def check(fn, *args):
        try:
            return fn(*args)
        except AssertionError as e:
            failures.append(str(e))

    for kind, ranges in c.cubes:
        cube, poly = make_cube(kind, c.nx, c.ny)
        nl = cube.shape[0]
        spline = L.spline_prepare(L.to_device(cube), L.INTERP_CUBIC)
        for prop in (True, False):
            _, path = warp_paths(name, prop)
            cell_path = path[warp_lanes(c.shape)[0]] if c.kernel != 'scalar' else np.full(xf.size, 'scalar')
            ref = MO.map_cube_fast(cube, xf[sub], yf[sub], 'cubic', propagate_nan=prop)
            evaluated = valid_cells(xf, yf, c.nx, c.ny, prop)
            xc, yc = np.nan_to_num(np.clip(xf, 0, c.nx - 1)), np.nan_to_num(np.clip(yf, 0, c.ny - 1))
            want = {l: np.where(evaluated, poly_eval(poly[l], xc, yc, c.nx, c.ny), np.nan) for l in poly}
            for begin, count in ranges:
                label = f'{name} {kind} planes ({begin}, {count}) propagate_nan={prop}'
                got_d = L.gather(spline, xd, yd, L.INTERP_CUBIC, plane_begin=begin, plane_count=count,
                                 propagate_nan=prop).reshape(count, -1)
                if c.kernel != 'scalar':
                    ref_d = scalar_launch(L, spline, xd, yd, c.nx, c.ny, begin, count, prop)
                    a, b = torch.nan_to_num(got_d, nan=-7.0), torch.nan_to_num(ref_d, nan=-7.0)
                    if not torch.equal(a, b):
                        failures.append(f'{label}: {int((a != b).sum())} voxels differ from the scalar kernel')
                got = got_d.cpu().numpy()
                rel = check(_rel_vs_scipy, got[:, sub], ref[begin:begin + count], label)
                poly_rel = np.zeros(got.shape)
                for l in poly:
                    if begin <= l < begin + count:
                        scale = float(np.max(np.abs(cube[l])))
                        r = check(_rel_vs_poly, got[l - begin], want[l], scale, f'{label} plane {l}')
                        poly_rel[l - begin] = r if r is not None else np.inf
                if (begin, count) == (0, nl) and rel is not None:
                    for p in np.unique(cell_path):
                        r = report.setdefault(f'propagate_nan={prop}', {}).setdefault(str(p),
                                                                                      {'scipy': 0.0, 'poly': 0.0})
                        on = cell_path == p
                        r['scipy'] = max(r['scipy'], float(rel[:, on[sub]].max(initial=0.0)))
                        r['poly'] = max(r['poly'], float(poly_rel[:, on].max(initial=0.0)))
    assert not failures, f'{len(failures)} disagreements:\n' + '\n'.join(failures[:40])
    write_parity_report(f'cubic_gather {name}', report)


@pytest.mark.gpu
@pytest.mark.timeout(120, method='thread')
def test_dense_launch_runs_the_mma_kernel_and_chunks_do_not(L):
    """The comparison above is only worth something if the two launches run different kernels."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    c = CASES_BY_NAME['12x9-rows-40']
    x, y, _ = build_map(c.name)
    xd, yd = L.to_device(x), L.to_device(y)
    cube, _ = make_cube('c3', c.nx, c.ny)
    spline = L.spline_prepare(L.to_device(cube), L.INTERP_CUBIC)
    torch.cuda.synchronize()

    def kernels(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == DeviceType.CUDA]

    dense = kernels(lambda: L.gather(spline, xd, yd, L.INTERP_CUBIC))
    chunked = kernels(lambda: scalar_launch(L, spline, xd, yd, c.nx, c.ny, 0, 3, True))
    if not dense and not chunked:
        pytest.skip('torch.profiler recorded no CUDA kernels on this machine')
    assert any(MMA_KERNEL in n for n in dense), dense
    assert not any(MMA_KERNEL in n for n in chunked) and any(SCALAR_KERNEL in n for n in chunked), chunked


@pytest.mark.gpu
@pytest.mark.timeout(120, method='thread')
def test_map_img_orthographic_40_takes_the_block_path(bc_hst):
    """The product path: BodyXY.map_img(interpolation='cubic') of the golden 7 x 10 disc onto a 40 x 40
    orthographic map (1600 cells >= 20 * 70: 4 x 8 cell blocks), the disc shifted partly out of the frame,
    against the oracle's map_img."""
    import planetmapper_b200 as pm
    from oracle import map_img_oracle as MO

    nx, ny = GOLDEN_DISC['nx'], GOLDEN_DISC['ny']
    body = pm.BodyXY(constants=bc_hst, nx=nx, ny=ny)
    body.set_disc_params(GOLDEN_DISC['x0'] - 1.5, GOLDEN_DISC['y0'] + 2.5, GOLDEN_DISC['r0'],
                         float(np.rad2deg(GOLDEN_DISC['rotation_radians'])))
    kw = dict(projection='orthographic', lon=body.subpoint_lon, lat=body.subpoint_lat, size=40)
    xm, ym = body.get_x_map(**kw), body.get_y_map(**kw)
    assert xm.shape == (40, 40) and select_kernel(xm.size, nx, ny, xm.shape[1]) == 'dense-2d'
    vis = np.isfinite(xm)
    with np.errstate(invalid='ignore'):
        out = vis & ((xm < 0) | (ym < 0) | (xm > nx - 1) | (ym > ny - 1))
    assert out.sum() > 50 and (vis & ~out).sum() > 200, (int(out.sum()), int(vis.sum()))
    cube = _cube(np.random.default_rng(4), 40, ny, nx)
    for prop in (True, False):
        got = body.map_img(cube, interpolation='cubic', propagate_nan=prop, **kw)
        want = MO.map_img(cube, xm, ym, 'cubic', propagate_nan=prop)
        rel = _rel_vs_scipy(got, want, f'map_img propagate_nan={prop}')
        assert np.isfinite(got).sum() > 1000, prop
        print(f'map_img orthographic 40 propagate_nan={prop}: worst rel vs scipy {rel.max():.2e}')
