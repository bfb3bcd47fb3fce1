"""
Frame constants for a TIME SERIES (BASELINE config C5: thousands of frames, a fresh
``BodyXY`` per epoch in the reference).

Once the per-pixel work takes ~40 microseconds per 1024 x 1024 frame on the GPU, the serial
host extraction of each frame's 92 constants (about 55 ephemeris / orientation evaluations,
~3 ms in Python, the same order through spiceypy: SURVEY.md 8(e) "limited only by serial
host constant extraction") is the whole cost of a series.  Epochs are independent, so the
extraction shards over host processes exactly like frames shard over GPUs: contiguous
blocks of epochs, no exchange, the SAME scalar code per epoch (``frame.build_body_constants``
+ ``frame.pack_frame``), hence bit-identical constants.  SPICE itself is not re-entrant
(SURVEY.md 8(b) "Threading"), which is why the workers are processes, each with its own
provider, and never threads.
"""
from __future__ import annotations

import atexit
import math
import os
import pickle
import struct
import subprocess
import sys

import numpy as np

from . import frame as F
from .shard import shard_range


def _block(provider, target, observer, ets, disc):
    """Frames (len(ets), 92) and km -> angular matrices (len(ets), 2, 2) of a block of epochs.  A disc value is a
    scalar shared by every epoch or an array holding one value per epoch of the block."""
    out = np.empty((len(ets), F.PMFRAME_NDOUBLES))
    k2a = np.empty((len(ets), 2, 2))
    for i, et in enumerate(ets):
        bc = F.build_body_constants(provider, target, None, observer, et=float(et), with_subsol=False)
        out[i] = F.pack_frame(bc, **{k: v[i] if isinstance(v, np.ndarray) else v for k, v in disc.items()})
        k2a[i] = F.km2angular_matrix(bc)
    return out, k2a


# ---- worker processes ---------------------------------------------------------------------
# Plain child interpreters running `python -m planetmapper_b200.series` and talking
# length-prefixed pickles over their pipes.  (multiprocessing's spawn / forkserver start
# methods re-import the caller's __main__, which breaks unguarded user scripts, and fork is not
# safe once the parent holds a CUDA context.)
def _send(stream, obj) -> None:
    data = pickle.dumps(obj, protocol=pickle.HIGHEST_PROTOCOL)
    stream.write(struct.pack('<Q', len(data)))
    stream.write(data)
    stream.flush()


def _recv(stream):
    head = stream.read(8)
    if len(head) < 8:
        raise EOFError('series worker closed its pipe')
    (n,) = struct.unpack('<Q', head)
    return pickle.loads(stream.read(n))


def _worker_main() -> None:
    import planetmapper_b200 as pm

    inp, out = sys.stdin.buffer, sys.stdout.buffer
    sys.stdout = sys.stderr  # stray prints must not corrupt the reply stream
    provider, provider_path = None, None
    while True:
        try:
            msg = _recv(inp)
        except EOFError:
            return
        try:
            kernel_path, target, observer, ets, disc, kepler = msg
            if provider is None or kernel_path != provider_path:   # the cached provider is keyed on its path
                pm.set_kernel_path(kernel_path)
                provider, provider_path = pm.get_default_provider(), kernel_path
            _send(out, ('ok', _block(_with_kepler(provider) if kepler else provider, target, observer, ets, disc)))
        except Exception as exc:  # reported to the parent, which raises
            _send(out, ('error', f'{type(exc).__name__}: {exc}'))


def _with_kepler(provider):
    """Analytic orbits for the bodies the kernels do not cover (minispice/kepler.py: BASELINE config C5 names
    Europa, which has no SPK segment in the bundled kernels)."""
    from .minispice.kepler import KeplerOrbitProvider

    return provider if isinstance(provider, KeplerOrbitProvider) else KeplerOrbitProvider(provider)


_WORKERS: list[subprocess.Popen] = []


def _workers(n: int) -> list[subprocess.Popen]:
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get('PYTHONPATH', ''),
               OMP_NUM_THREADS='1', OPENBLAS_NUM_THREADS='1', MKL_NUM_THREADS='1')
    _WORKERS[:] = [w for w in _WORKERS if w.poll() is None]
    while len(_WORKERS) < n:
        _WORKERS.append(subprocess.Popen([sys.executable, '-m', 'planetmapper_b200.series'], stdin=subprocess.PIPE,
                                         stdout=subprocess.PIPE, env=env))
    return _WORKERS[:n]


def shutdown_pool() -> None:
    """Stop the worker processes (they are otherwise kept for the next series)."""
    for w in _WORKERS:
        try:
            w.stdin.close()
            w.wait(timeout=10)
        except Exception:
            w.kill()
    _WORKERS.clear()


atexit.register(shutdown_pool)


def default_workers() -> int:
    """Host processes to use: the cores this process may run on, shared between the ranks
    of a torchrun job (LOCAL_WORLD_SIZE)."""
    total = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        cores = total
    if cores < total:   # this rank already owns a slice of the host (shard.bind_rank_to_cores, taskset, cgroups)
        return max(1, cores)
    ranks = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))
    return max(1, cores // ranks)


def _disc_value(name: str, value, n: int):
    """A disc parameter as given (a scalar, shared by every epoch) or as a float64 array of one value per epoch."""
    arr = np.asarray(value, dtype=np.float64)
    if arr.ndim == 0:
        if not np.isfinite(arr):
            raise ValueError(f'{name} must be finite')
        return value
    if arr.shape != (n,):
        raise ValueError(f'{name} must be a scalar or hold one value per epoch ({n}), not shape {arr.shape}')
    if not np.all(np.isfinite(arr)):
        raise ValueError(f'{name} must be finite at every epoch')
    return np.ascontiguousarray(arr)


def build_series_frames(target, ets, observer='EARTH', *, nx: int, ny: int, x0, y0, r0,
                        rotation_radians=0.0, alt: float = 0.0, workers: int | None = None, provider=None,
                        kepler: bool = False, with_km2angular: bool = False):
    """PMFrame constants, shape (len(ets), 92), for ``target`` seen from ``observer`` at the
    ephemeris times ``ets``.

    ``x0``, ``y0``, ``r0`` and ``rotation_radians`` are each a scalar shared by every epoch or an array of
    ``len(ets)`` values, one per epoch (pointing drift, ``r0`` following the distance at a fixed plate scale):
    frame f is ``pack_frame(constants_f, x0=x0[f], ...)``.  ``nx``, ``ny`` and ``alt`` are shared.
    ``workers`` host processes (default: :func:`default_workers`) each take one contiguous
    block of epochs; ``workers <= 1``, a short series, or an explicit in-process ``provider``
    runs serially in this process.  The result does not depend on ``workers``.  ``kepler=True`` answers
    the ephemeris of bodies without SPK coverage from the analytic orbits of ``minispice/kepler.py``
    (synthetic positions: Europa of BASELINE config C5).  ``with_km2angular=True`` returns
    ``(frames, km2angular)``, the second the (len(ets), 2, 2) km -> angular matrices of the epochs
    (Body._get_km2angular_matrix), which :func:`transform` needs for km -> angular in a custom angular frame.
    """
    import planetmapper_b200 as pm

    ets = np.asarray(ets, dtype=np.float64).reshape(-1)
    disc = dict(nx=nx, ny=ny, alt=alt)
    for name, value in (('x0', x0), ('y0', y0), ('r0', r0), ('rotation_radians', rotation_radians)):
        disc[name] = _disc_value(name, value, len(ets))
    workers = default_workers() if workers is None else int(workers)
    workers = min(workers, max(1, len(ets) // 16))   # a block under ~16 epochs does not pay for the hand-off
    if pm.provider_is_custom():   # an in-process provider cannot be rebuilt inside a worker
        workers = 1
    if provider is not None or workers <= 1:
        prov = provider if provider is not None else pm.get_default_provider()
        frames, k2a = _block(_with_kepler(prov) if kepler else prov, target, observer, ets, disc)
        return (frames, k2a) if with_km2angular else frames
    procs = _workers(workers)
    try:
        for w, proc in enumerate(procs):
            part = slice(*shard_range(len(ets), w, workers))
            block_disc = {k: v[part] if isinstance(v, np.ndarray) else v for k, v in disc.items()}
            _send(proc.stdin, (pm._KERNEL_PATH, str(target), str(observer), ets[part], block_disc, bool(kepler)))
        replies = [_recv(proc.stdout) for proc in procs]   # every reply is drained before any error is raised
    except BaseException:
        shutdown_pool()   # a dead or half-read worker must not serve the next call
        raise
    failed = [payload for status, payload in replies if status != 'ok']
    if failed:
        raise RuntimeError(f'series worker failed: {failed[0]}')
    frames = np.concatenate([payload[0] for _, payload in replies], axis=0)
    if with_km2angular:
        return frames, np.concatenate([payload[1] for _, payload in replies], axis=0)
    return frames


def iter_backplane_batches(frames: np.ndarray, nx: int, ny: int, names, batch: int = 32):
    """Backplane images of a series, ``batch`` frames per fused launch.

    Yields ``(first, planes)`` with ``planes`` a CUDA tensor of shape
    ``(n, len(set(names)), ny, nx)`` holding frames ``first .. first + n`` (planes in
    backplane-registration order, like ``BodyXY.get_backplane_imgs``).  The tensor is REUSED by
    the next iteration (a 4096-frame series of 12 planes would be 412 GB): consume or copy it
    before advancing.  Equivalent to ``BodyXY(target, utc_i, ...).get_backplane_img(name)`` for
    every epoch and name in the reference (body_xy.py:2586), one launch per batch instead of one
    Python loop per pixel, stage and frame.
    """
    from . import _lib as L

    torch = L._torch()
    mask = L.mask_from_names([str(n).strip().upper() for n in names])
    fd = L.to_device(np.ascontiguousarray(frames, dtype=np.float64))
    out = torch.empty((min(batch, len(frames)), L.popcount(mask), ny, nx), dtype=torch.float64, device=fd.device)
    for first in range(0, len(frames), batch):
        n = min(batch, len(frames) - first)
        L.backplanes_img(fd[first:first + n], nx, ny, mask, out=out[:n])
        yield first, out[:n]


def map_series(frames: np.ndarray, imgs, nx: int, ny: int, lons, lats, *, interpolation='linear',
               propagate_nan: bool = True, batch: int = 32, out=None):
    """``BodyXY(...).map_img(img_f, ...)`` for every frame f of a series (body_xy.py:1414-1631 once per
    epoch in the reference): frame f's image is mapped onto the lon / lat grid with frame f's own
    disc geometry.  Per batch of frames: ONE launch for all x / y maps (``pm_backplanes_map_batch``),
    the NaN repair of the batch's images (linear), ONE grouped gather of one image per map.

    ``imgs``: (n_frames, ny, nx) array or tensor; a stack that is not a float64 CUDA tensor is uploaded and
    converted one batch at a time.  ``lons`` / ``lats``: the map grid (degrees, e.g. from
    ``generate_map_coordinates``); ``interpolation``: 'nearest' or 'linear'.  Returns a CUDA tensor
    (n_frames,) + grid shape (``out`` if given).  :func:`iter_mapped_series` maps with every interpolating
    spline degree, and a cube per epoch.
    """
    from . import _lib as L

    torch = L._torch()
    mode = {'nearest': L.INTERP_NEAREST, 'linear': L.INTERP_LINEAR, 1: L.INTERP_LINEAR}.get(interpolation)
    if mode is None:
        raise NotImplementedError("map_series: interpolation must be 'nearest' or 'linear'")
    frames = np.ascontiguousarray(frames, dtype=np.float64)
    if not isinstance(imgs, torch.Tensor):
        imgs = np.asarray(imgs)
    if tuple(imgs.shape) != (len(frames), ny, nx):
        raise ValueError(f'imgs must have shape ({len(frames)}, {ny}, {nx})')
    lons, lats = np.asarray(lons, dtype=np.float64), np.asarray(lats, dtype=np.float64)
    if out is None:
        out = torch.empty((len(frames),) + lons.shape, dtype=torch.float64, device='cuda')
    for first, n, xy, src, stride in _prepared_batches(frames, imgs, nx, ny, lons, lats, mode, batch,
                                                       L.mask_from_names(['PIXEL-X', 'PIXEL-Y']), 1):
        L.gather_grouped(src, xy[:, 0], xy[:, 1], mode, 1, stride, propagate_nan=propagate_nan,
                         out=out[first:first + n])
    return out


SERIES_MEMORY_SHARE = 0.4   # of the free device memory, for a batch's cubes, prepared operand, maps and output


def iter_mapped_series(frames: np.ndarray, cubes, nx: int, ny: int, lons, lats, *, interpolation='linear',
                       spline_smoothing: float = 0, propagate_nan: bool = True, batch: int | None = None):
    """``Observation(data=cube_f, ...).get_mapped_data(interpolation)`` (``BodyXY.map_img`` for an image) for every
    epoch f of a series, each with frame f's own geometry and disc, in batches of epochs.

    ``cubes``: (n_frames, nλ, ny, nx) or (n_frames, ny, nx) (one image per epoch), a numpy array or a CUDA
    tensor; host input is uploaded one batch at a time.  ``lons`` / ``lats``: the map grid shared by every epoch
    (degrees, e.g. from ``generate_map_coordinates``).  ``interpolation``: everything map_img accepts without
    smoothing ('nearest', 'linear', 'quadratic', 'cubic', a degree 1..3 or a (k_rows, k_cols) pair), with
    map_img's errors; 'smooth' and ``spline_smoothing != 0`` raise NotImplementedError.

    Yields ``(first, mapped)``: ``mapped`` is a CUDA tensor (n, nλ) + grid shape ((n,) + grid shape for 3-D
    input) holding epochs first .. first + n, equal to the single-epoch call bit for bit.  The tensor is REUSED
    by the next iteration: consume or copy it before advancing.  Per batch: one launch for every epoch's x / y
    map, one spline preparation of the whole batch and one grouped gather (a cube series of cubic maps with
    >= 20 map cells per image pixel: pm_gather's dense-map kernel once per epoch).  ``batch`` (epochs per batch)
    defaults to what keeps a batch within SERIES_MEMORY_SHARE of the free device memory.
    """
    mode, frames, lons, lats = _series_args('iter_mapped_series', frames, cubes, nx, ny, lons, lats, interpolation,
                                            spline_smoothing, batch)
    return _mapped_series(frames, cubes, nx, ny, lons, lats, mode, propagate_nan, batch)


def _series_args(fn, frames, cubes, nx, ny, lons, lats, interpolation, spline_smoothing, batch):
    """The argument rules of the mapped-series functions, checked before any device work: (mode, frames, lons,
    lats) as the batches need them."""
    from .body_xy import _interpolation_mode

    if interpolation == 'smooth' or spline_smoothing != 0:
        raise NotImplementedError(f"{fn}: 'smooth' and smoothing splines (spline_smoothing != 0) fit "
                                  'per-epoch grids; map those epochs with Observation.get_mapped_data')
    mode = _interpolation_mode(interpolation, 0)
    frames = np.ascontiguousarray(frames, dtype=np.float64)
    if frames.ndim != 2 or frames.shape[1] != F.PMFRAME_NDOUBLES:
        raise ValueError(f'frames must have shape (n_frames, {F.PMFRAME_NDOUBLES})')
    shape = tuple(int(d) for d in cubes.shape)
    if len(shape) not in (3, 4) or shape[0] != len(frames) or shape[-2:] != (ny, nx) or 0 in shape[1:]:
        raise ValueError(f'cubes must have shape ({len(frames)}, nλ, {ny}, {nx}) or ({len(frames)}, {ny}, {nx}), '
                         f'not {shape}')
    lons, lats = np.asarray(lons, dtype=np.float64), np.asarray(lats, dtype=np.float64)
    if lons.shape != lats.shape or lons.size == 0:
        raise ValueError(f'lons and lats must have one shape, not {lons.shape} and {lats.shape}')
    if batch is not None and int(batch) < 1:
        raise ValueError('batch must be at least 1')
    return mode, frames, lons, lats


def _series_stride(n_planes: int, mode: int) -> int:
    """Planes per epoch in the prepared cube: a spline cube of several planes starts every epoch on a plane quad
    (the gather reads quads); one image per epoch, or the raw cube of nearest, is packed as given."""
    from . import _lib as L

    return n_planes if mode == L.INTERP_NEAREST or n_planes == 1 else (n_planes + 3) // 4 * 4


def _prepared_batches(frames, cubes, nx, ny, lons, lats, mode, batch, mask, out_planes):
    """The batches of a mapped series: per batch of n epochs ONE pm_backplanes_map_batch launch with the planes of
    ``mask`` and the batch's cubes staged at ``_series_stride`` planes per epoch (pad planes all NaN) and prepared
    once (nearest reads the staged cube as it is).  Yields ``(first, n, maps, src, stride)``: maps (n,
    popcount(mask)) + grid and the gather source, both REUSED by the next batch.  ``batch`` None: what keeps a
    batch's cubes, prepared operand, maps and ``out_planes`` output planes per epoch within SERIES_MEMORY_SHARE of
    the free device memory."""
    from . import _lib as L

    torch = L._torch()
    lib = L.load_library()
    n_frames = len(frames)
    nl = 1 if cubes.ndim == 3 else int(cubes.shape[1])
    stride = _series_stride(nl, mode)
    n_cells = lons.size
    n_maps = L.popcount(mask)
    # the prepare launches put a plane per grid row (<= 65535), the map and gather launches an epoch per grid row
    limit = 65535 // stride
    if batch is None:
        per_frame = 8 * (out_planes + n_maps) * n_cells + 8 * stride * ny * nx   # output, maps, uploaded cube
        if mode != L.INTERP_NEAREST:
            per_frame += (lib.pm_spline_coef_bytes(stride, ny, nx) + lib.pm_spline_nanbits_bytes(stride, ny, nx) +
                          lib.pm_spline_work_bytes(stride, ny, nx, mode))
        free, _total = torch.cuda.mem_get_info()
        budget = int(SERIES_MEMORY_SHARE * free)
        if per_frame > budget:
            raise ValueError(f'one epoch needs {per_frame / 1e9:.1f} GB of device memory and {budget / 1e9:.1f} GB '
                             'are available to a batch: map that epoch with Observation.iter_mapped_data')
        batch = budget // per_frame
    batch = int(max(1, min(batch, n_frames, limit)))
    fd = L.to_device(frames)
    lod = L.to_device(lons % 360)
    lad = L.to_device(lats)
    maps = torch.empty((batch, n_maps) + lons.shape, dtype=torch.float64, device=fd.device)
    on_device = isinstance(cubes, torch.Tensor) and cubes.is_cuda and cubes.dtype == torch.float64
    staged = None
    if stride != nl or not on_device:
        # the batch's cubes at `stride` planes per epoch; pad planes are all NaN and are never mapped
        staged = torch.full((batch, stride, ny, nx), float('nan'), dtype=torch.float64, device=fd.device)
    for first in range(0, n_frames, batch):
        n = min(batch, n_frames - first)
        L.backplanes_map_batch(fd[first:first + n], lod, lad, mask, out=maps[:n])
        part = cubes[first:first + n]
        if staged is None:
            cube = part.reshape(n * nl, ny, nx).contiguous()
        else:
            if not isinstance(part, torch.Tensor):
                part = torch.from_numpy(np.ascontiguousarray(part, dtype=np.float64))
            staged[:n, :nl].copy_(part.reshape(n, nl, ny, nx))
            cube = staged[:n].view(n * stride, ny, nx)
        yield first, n, maps[:n], (cube if mode == L.INTERP_NEAREST else L.spline_prepare(cube, mode)), stride


def _mapped_series(frames, cubes, nx, ny, lons, lats, mode, propagate_nan, batch):
    from . import _lib as L

    torch = L._torch()
    nl = 1 if cubes.ndim == 3 else int(cubes.shape[1])
    out = None
    for first, n, xy, src, stride in _prepared_batches(frames, cubes, nx, ny, lons, lats, mode, batch,
                                                       L.mask_from_names(['PIXEL-X', 'PIXEL-Y']), nl):
        if out is None:   # the first batch is a full one
            out = torch.empty((n, nl) + lons.shape, dtype=torch.float64, device=xy.device)
        L.gather_grouped(src, xy[:, 0], xy[:, 1], mode, nl, stride, propagate_nan=propagate_nan, out=out[:n])
        yield first, (out[:n, 0] if cubes.ndim == 3 else out[:n])


def composite_mapped_series(frames: np.ndarray, cubes, nx: int, ny: int, lons, lats, *, interpolation='linear',
                            spline_smoothing: float = 0, propagate_nan: bool = True, method: str = 'mean',
                            max_emission=None, batch: int | None = None):
    """The epochs of a mapped series combined into ONE map on the device: a composite of many observations of one
    target on a shared lon / lat grid (frames spread over a rotation, the tiles or dithers of a mosaic: one epoch
    repeated with different discs).  Takes what :func:`iter_mapped_series` takes, with its errors.

    Let v_f be the value :func:`iter_mapped_series` produces for epoch f at a plane and cell, and e_f epoch f's
    EMISSION angle at that cell (``BodyXY.get_backplane_map('EMISSION')``).  Epoch f contributes there iff v_f is
    not NaN and, when ``max_emission`` (degrees, 0..180) is given, e_f <= max_emission (a NaN e_f does not).

    ``method='mean'``: the contributions summed in epoch order by IEEE adds, over their count (``np.nanmean`` with
    that summation order); tag = the count.  ``method='min_emission'``: the contribution of the epoch with the
    smallest e_f, ties to the lowest epoch; tag = that epoch's index.  The choice is per voxel: a NaN pixel of the
    best epoch in one plane falls through to the next-best epoch for that plane.  Cells without a contribution
    are NaN with tag 0 (mean) or -1 (min_emission).

    Returns ``(composite, tag)``: CUDA tensors (nλ,) + grid shape (grid shape for 3-D input), float64 and int32.
    Per batch of epochs: one map launch (PIXEL-X / PIXEL-Y, plus EMISSION when the method or the cut reads it), the
    spline preparation of :func:`iter_mapped_series` and ONE pm_composite_grouped launch, which folds every
    epoch's voxels into accumulators held in registers and never stores the per-epoch maps.  The result does not
    depend on ``batch``, bit for bit.  Every mode equals the fold of :func:`iter_mapped_series`' output bit for
    bit, except cubic cubes on maps of >= 20 cells per image pixel, where that function runs the DMMA gather and
    the values may differ in the last bits.
    """
    from . import _lib as L

    mode, frames, lons, lats = _series_args('composite_mapped_series', frames, cubes, nx, ny, lons, lats,
                                            interpolation, spline_smoothing, batch)
    if method not in L.COMPOSITE_METHODS:
        raise ValueError(f"method must be one of {sorted(L.COMPOSITE_METHODS)}, not {method!r}")
    if max_emission is not None:
        max_emission = float(max_emission)
        if not 0.0 <= max_emission <= 180.0:
            raise ValueError(f'max_emission must be None or an angle in [0, 180] degrees, not {max_emission}')
    if len(frames) == 0:
        raise ValueError('composite_mapped_series needs at least one epoch')
    torch = L._torch()
    nl = 1 if cubes.ndim == 3 else int(cubes.shape[1])
    shape = (nl,) + lons.shape
    value = torch.empty(shape, dtype=torch.float64, device='cuda')
    tag = torch.empty(shape, dtype=torch.int32, device='cuda')
    key = torch.empty(shape, dtype=torch.float64, device='cuda') if method == 'min_emission' else None
    # a plain mean keeps the x / y-only mask (the map kernel's fixed-plane-set instantiation)
    names = ['PIXEL-X', 'PIXEL-Y'] + (['EMISSION'] if method == 'min_emission' or max_emission is not None else [])
    cut = float('inf') if max_emission is None else max_emission
    for first, n, maps, src, stride in _prepared_batches(frames, cubes, nx, ny, lons, lats, mode, batch,
                                                         L.mask_from_names(names), 0):
        L.composite_grouped(src, maps, mode, nl, stride, method, value, tag, key=key, max_emission=cut,
                            epoch_begin=first, first=first == 0, last=first + n == len(frames),
                            propagate_nan=propagate_nan)
    return (value[0], tag[0]) if cubes.ndim == 3 else (value, tag)


# ---- point transforms over the epochs of a series -------------------------------------------------
_SOURCES = ('xy', 'angular', 'km', 'radec', 'lonlat')


def frames_at_alt(frames: np.ndarray, alt: float) -> np.ndarray:
    """The frames of a series (built with ``alt=0``) with the target's radii raised by ``alt`` km: per epoch the
    radii, ``re``, ``f`` and ``r_eq`` that ``pack_frame(..., alt=alt)`` writes, with the same operations
    (BodyXY._frame_dev(alt), the reference's _AdjustedSurfaceAltitude).  ``r_cut2``, the image kernels'
    early-out radius, keeps its value: no point transform reads it."""
    out = np.array(frames, dtype=np.float64, copy=True)
    o = F.PMFRAME_OFFSETS
    radii = out[:, o['radii'][0]:o['radii'][0] + 3] + float(alt)
    re, rp = radii[:, 0].copy(), radii[:, 2].copy()
    out[:, o['radii'][0]:o['radii'][0] + 3] = radii
    out[:, o['re'][0]] = re
    out[:, o['f'][0]] = (re - rp) / re
    out[:, o['r_eq'][0]] = re
    return out


def _angular_table(frames, origin_ra, origin_dec, coordinate_rotation, km2angular) -> np.ndarray:
    """(n_frames, 13) rows of BodyXY._angular_aux, one per epoch: the obsvec -> angular matrix centred on
    (origin_ra, origin_dec), each defaulting to THAT epoch's target RA / Dec (from its P0, as
    build_body_constants derives them), then the epoch's km -> angular matrix (NaN when not given: only a
    km source reads it)."""
    o = F.PMFRAME_OFFSETS['P0'][0]
    table = np.full((len(frames), 13), np.nan)
    for f in range(len(frames)):
        _, ra, dec = F._recrad(frames[f, o:o + 3])
        m = F.obsvec2angular_matrix(math.degrees(ra) if origin_ra is None else float(origin_ra),
                                    math.degrees(dec) if origin_dec is None else float(origin_dec),
                                    float(coordinate_rotation))
        table[f, :9] = m.ravel()
        if km2angular is not None:
            table[f, 9:] = km2angular[f].ravel()
    return table


def transform(frames, src: str, dst: str, a, b, *, alt: float = 0.0, not_visible_nan: bool = False,
              not_found_nan: bool = True, planetocentric: bool = False, origin_ra=None, origin_dec=None,
              coordinate_rotation: float = 0.0, per_frame: bool = False, km2angular=None):
    """Points (a, b) of coordinate system ``src`` in system ``dst`` at every epoch of a series, in one launch:
    row f is what ``BodyXY`` with frame f's epoch and disc parameters returns from the matching method
    (``xy2lonlat``, ``lonlat2xy``, ``xy2radec``, ``km2angular``, ...), bit for bit.

    ``frames``: (n_frames, 92) from :func:`build_series_frames` (``alt=0``).  ``src``: 'xy', 'angular', 'km',
    'radec' or 'lonlat'; ``dst`` also 'centric' (planetocentric lon / lat, graphic2centric_lonlat);
    'lonlat' -> 'lonlat' with ``planetocentric=True`` is centric2graphic_lonlat.  ``a`` / ``b`` broadcast like
    the BodyXY methods' inputs and are shared by every epoch; with ``per_frame=True`` their leading axis is the
    epoch (e.g. a tracked pixel per frame).  ``alt``, ``not_visible_nan``, ``not_found_nan``, ``planetocentric``
    and the angular-frame arguments mean what they mean for the BodyXY method; ``origin_ra`` / ``origin_dec``
    default to each epoch's own target RA / Dec.  km -> angular in a custom angular frame also needs
    ``km2angular``, the (n_frames, 2, 2) matrices of ``build_series_frames(..., with_km2angular=True)``.
    ``not_found_nan=False`` raises NotFoundError, naming the first epoch, when a ray misses the target.

    Returns two float64 CUDA tensors shaped (n_frames,) + point shape.
    """
    from . import _lib as L
    from .body_xy import BodyXY, NotFoundError

    frames = np.ascontiguousarray(frames, dtype=np.float64)
    if frames.ndim != 2 or frames.shape[1] != F.PMFRAME_NDOUBLES or len(frames) == 0:
        raise ValueError(f'frames must have shape (n_frames, {F.PMFRAME_NDOUBLES}) with n_frames >= 1')
    n_frames = len(frames)
    if src not in _SOURCES or dst not in L.COORD:
        raise ValueError(f'unknown coordinate pair {src!r} -> {dst!r}')
    if src == dst and src != 'lonlat':
        raise ValueError(f'{src!r} -> {dst!r} is not a transform')
    custom_angular = not (origin_ra is None and origin_dec is None and coordinate_rotation == 0.0)
    if custom_angular and 'angular' not in (src, dst):
        raise ValueError('origin_ra / origin_dec / coordinate_rotation only apply to the angular system')
    if custom_angular and src == 'km':
        if km2angular is None:
            raise ValueError('km -> angular in a custom angular frame needs the epochs\' km2angular matrices '
                             '(build_series_frames(..., with_km2angular=True))')
        km2angular = np.asarray(km2angular, dtype=np.float64)
        if km2angular.shape != (n_frames, 2, 2):
            raise ValueError(f'km2angular must have shape ({n_frames}, 2, 2)')
    aa, bb = np.broadcast_arrays(np.asarray(a, dtype=float), np.asarray(b, dtype=float))
    if per_frame and (aa.ndim == 0 or aa.shape[0] != n_frames):
        raise ValueError(f'per_frame points need a leading axis of {n_frames} epochs, not shape {aa.shape}')
    shape = (n_frames,) + (aa.shape[1:] if per_frame else aa.shape)

    # each public method's own host rules (BodyXY.xy2lonlat / lonlat2xy / _transform)
    alt = float(alt)
    xy2lonlat = src == 'xy' and dst == 'lonlat'
    if xy2lonlat or (not math.isfinite(alt) and dst in ('lonlat', 'centric')):
        BodyXY._check_alt(alt)
    if not math.isfinite(alt):   # Body._lonlat2targvec_radians: non-finite alt -> NaN
        torch = L._torch()
        nan = torch.full(shape, float('nan'), dtype=torch.float64, device='cuda')
        return nan, nan.clone()
    fd = L.to_device(frames)
    a_dev, b_dev = L.to_device(aa), L.to_device(bb)   # scalars arrive as one point: outputs are reshaped below
    if xy2lonlat and not planetocentric:
        fa = L.to_device(frames_at_alt(frames, alt)) if alt != 0.0 else fd
        lon, lat, missed = L.xy2lonlat_batch(fa, a_dev, b_dev, per_frame=per_frame)
        if not not_found_nan:
            n = int(np.prod(shape[1:]))   # BodyXY.xy2lonlat: a missed ray, or NaN at a finite input
            finite_in = (a_dev.isfinite() & b_dev.isfinite()).reshape(n_frames if per_frame else 1, n)
            bad = (missed > 0) | (finite_in & lon.reshape(n_frames, n).isnan()).any(dim=1)
            _raise_first_epoch(bad, NotFoundError)
        return lon.reshape(shape), lat.reshape(shape)
    if src == 'lonlat' and dst == 'xy':
        x, y = L.lonlat2xy_batch(fd, a_dev, b_dev, per_frame=per_frame, not_visible_nan=not_visible_nan, alt=alt,
                                 planetocentric=planetocentric)
        return x.reshape(shape), y.reshape(shape)
    # a lon / lat destination intersects the ellipsoid raised by alt (_AdjustedSurfaceAltitude)
    if dst in ('lonlat', 'centric') and src != 'lonlat' and alt != 0.0:
        fd = L.to_device(frames_at_alt(frames, alt))
    aux = None
    if custom_angular:
        aux = L.to_device(_angular_table(frames, origin_ra, origin_dec, coordinate_rotation, km2angular))
    oa, ob, missed = L.transform_batch(fd, src, dst, a_dev, b_dev, per_frame=per_frame, alt=alt,
                                       not_visible_nan=not_visible_nan, planetocentric=planetocentric, aux13_dev=aux)
    if not not_found_nan:
        _raise_first_epoch(missed > 0, NotFoundError)
    return oa.reshape(shape), ob.reshape(shape)


def _raise_first_epoch(bad, error) -> None:
    """``error`` naming the first epoch flagged in the (n_frames,) bool CUDA tensor ``bad``."""
    bad = bad.cpu().numpy()
    if bad.any():
        raise error(f'ray does not intercept the target body (epoch {int(np.argmax(bad))})')


if __name__ == '__main__':
    _worker_main()
