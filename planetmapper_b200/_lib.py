"""
ctypes binding of libpm_b200.so (C ABI: include/pm_b200.h) plus thin wrappers that
take and return torch CUDA tensors.  PyTorch is used for device memory and streams
only; all arithmetic happens in the hand-written sm_100a kernels.

There is NO CPU fallback: if the library is missing, or no CUDA device is visible,
the wrappers raise :class:`PMLibraryError`.
"""

from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('PM_B200_LIBRARY') or os.path.join(_HERE, 'libpm_b200.so')

N_PLANES = 26
ALL_PLANES = (1 << N_PLANES) - 1
INTERP_NEAREST, INTERP_LINEAR, INTERP_QUADRATIC, INTERP_CUBIC = 0, 1, 2, 3
INTERP_MIXED = 0x100   # | degree along rows << 4 | degree along columns
PROJ_ORTHOGRAPHIC, PROJ_AZIMUTHAL, PROJ_AZIMUTHAL_EQUAL_AREA = 1, 2, 3
FLAG_NOT_VISIBLE_NAN = 1
FLAG_PROPAGATE_NAN = 2
FLAG_PLANETOCENTRIC = 4
FLAG_RING_ALL = 8

PLANE_NAMES = [
    'LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'RA', 'DEC', 'PIXEL-X',
    'PIXEL-Y', 'KM-X', 'KM-Y', 'ANGULAR-X', 'ANGULAR-Y', 'PHASE', 'INCIDENCE',
    'EMISSION', 'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER',
    'LIMB-DISTANCE', 'LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC', 'RING-RADIUS',
    'RING-LON-GRAPHIC', 'RING-DISTANCE',
]
PLANE_ID = {n: i for i, n in enumerate(PLANE_NAMES)}

# every symbol include/pm_b200.h declares
EXPORTED_SYMBOLS = [
    'pm_abi_version', 'pm_error_string', 'pm_launch_count', 'pm_backplanes_img',
    'pm_backplanes_map', 'pm_backplanes_map_host', 'pm_xy2lonlat', 'pm_lonlat2xy', 'pm_lonlat2xy_alt', 'pm_proj_inverse', 'pm_gather',
    'pm_spline_coef_bytes', 'pm_spline_nanbits_bytes', 'pm_spline_planebits_bytes',
    'pm_spline_work_bytes', 'pm_spline_prepare', 'pm_fp64_peak_probe', 'pm_math_probe',
    'pm_nan_minmax', 'pm_pchip_work_bytes', 'pm_pchip_resample', 'pm_gather_grid_linear',
    'pm_fits_data_unit_bytes', 'pm_fits_stage', 'pm_backplanes_map_batch', 'pm_gather_paired',
    'pm_host_ssb_state', 'pm_host_orientation', 'pm_backplanes_img_host', 'pm_transform', 'pm_fp64_probe', 'pm_proj_forward',
    'pm_backplanes_points_host', 'pm_regrid_work_bytes', 'pm_regrid_fit', 'pm_gather_regrid',
    'pm_xy2lonlat_batch', 'pm_lonlat2xy_batch', 'pm_transform_batch', 'pm_gather_grouped',
]


class PMLibraryError(RuntimeError):
    """The CUDA library is missing, failed to load, or reported an error."""


_lib = None


def load_library() -> ctypes.CDLL:
    """Load libpm_b200.so (no compute; works without a GPU)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PMLibraryError(
            f'{LIB_PATH} not found: build it with `make -C planetmapper_b200/csrc` or '
            '`python -c "import __graft_entry__ as g; g.build()"`. There is no CPU fallback.'
        )
    lib = ctypes.CDLL(LIB_PATH)
    c_i, c_i64, c_u64, c_u32, c_p = (ctypes.c_int, ctypes.c_int64, ctypes.c_uint64,
                                     ctypes.c_uint32, ctypes.c_void_p)
    lib.pm_abi_version.restype = c_i
    lib.pm_error_string.restype = ctypes.c_char_p
    lib.pm_error_string.argtypes = [c_i]
    lib.pm_launch_count.restype = c_u64
    lib.pm_backplanes_img.argtypes = [c_p, c_i, c_i, c_i, c_u64, c_p, c_p]
    lib.pm_backplanes_map.argtypes = [c_p, c_p, c_p, c_i64, c_u64, c_p, c_p]
    lib.pm_backplanes_map_host.argtypes = [c_p, c_p, c_p, c_i64, c_u64, c_p, c_p]
    lib.pm_backplanes_img_host.argtypes = [c_p, c_i, c_i, c_u64, c_p, c_p]
    lib.pm_backplanes_img_host.restype = c_i
    lib.pm_backplanes_points_host.argtypes = [c_p, c_p, c_p, c_i64, c_u64, c_u32, c_p, c_p]
    lib.pm_backplanes_points_host.restype = c_i
    lib.pm_transform.argtypes = [c_p, c_i, c_i, c_p, c_p, c_i64, ctypes.c_double, c_u32, c_p, c_p, c_p, c_p, c_p]
    lib.pm_transform.restype = c_i
    lib.pm_xy2lonlat.argtypes = [c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p]
    lib.pm_lonlat2xy.argtypes = [c_p, c_p, c_p, c_i64, c_u32, c_p, c_p, c_p]
    lib.pm_lonlat2xy_alt.argtypes = [c_p, c_p, c_p, c_i64, ctypes.c_double, c_u32, c_p, c_p, c_p]
    lib.pm_xy2lonlat_batch.argtypes = [c_p, c_i, c_p, c_p, c_i64, c_i64, c_p, c_p, c_p, c_p]
    lib.pm_lonlat2xy_batch.argtypes = [c_p, c_i, c_p, c_p, c_i64, c_i64, ctypes.c_double, c_u32, c_p, c_p, c_p]
    lib.pm_transform_batch.argtypes = [c_p, c_i, c_i, c_i, c_p, c_p, c_i64, c_i64, ctypes.c_double, c_u32, c_p, c_p,
                                       c_p, c_p, c_p]
    for fn in ('pm_xy2lonlat_batch', 'pm_lonlat2xy_batch', 'pm_transform_batch'):
        getattr(lib, fn).restype = c_i
    lib.pm_proj_inverse.argtypes = [c_i, c_p, c_p, c_p, c_i64, c_p, c_p, c_p]
    lib.pm_proj_forward.argtypes = [c_i, c_p, c_p, c_p, c_i64, c_p, c_p, c_p]
    lib.pm_proj_forward.restype = c_i
    lib.pm_gather.argtypes = [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_i64, c_i64, c_i, c_u32,
                              c_p, c_p]
    for fn in ('pm_spline_coef_bytes', 'pm_spline_nanbits_bytes', 'pm_spline_work_bytes',
               'pm_spline_planebits_bytes'):
        getattr(lib, fn).restype = c_i64
    lib.pm_spline_coef_bytes.argtypes = [c_i, c_i, c_i]
    lib.pm_spline_nanbits_bytes.argtypes = [c_i, c_i, c_i]
    lib.pm_spline_planebits_bytes.argtypes = [c_i]
    lib.pm_spline_work_bytes.argtypes = [c_i, c_i, c_i, c_i]
    lib.pm_spline_prepare.argtypes = [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p]
    lib.pm_regrid_work_bytes.restype = c_i64
    lib.pm_regrid_work_bytes.argtypes = [c_i, c_i, c_i, c_i, c_i]
    lib.pm_regrid_fit.restype = c_i
    lib.pm_regrid_fit.argtypes = [c_p, c_p, c_i, c_i, c_i, c_i, c_i, ctypes.c_double, c_i, c_p, c_p, c_p, c_p, c_p,
                                  c_p, c_p, c_p]
    lib.pm_gather_regrid.restype = c_i
    lib.pm_gather_regrid.argtypes = [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_i64,
                                     c_u32, c_p, c_p]
    lib.pm_fp64_peak_probe.argtypes = [c_i, c_p, c_p]
    lib.pm_fp64_probe.argtypes = [c_i, c_i, c_p, c_p]
    lib.pm_fp64_probe.restype = c_i
    lib.pm_math_probe.argtypes = [c_i, c_p, c_p, c_i64, c_p, c_p]
    lib.pm_nan_minmax.argtypes = [c_p, c_i64, c_p, c_p]
    lib.pm_pchip_work_bytes.restype = c_i64
    lib.pm_pchip_work_bytes.argtypes = [c_i, c_i, c_i, c_i]
    lib.pm_pchip_resample.argtypes = [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p]
    lib.pm_gather_grid_linear.argtypes = [c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_i, c_i, c_p, c_p, c_i64,
                                          c_u32, c_p, c_p]
    lib.pm_fits_data_unit_bytes.restype = c_i64
    lib.pm_fits_data_unit_bytes.argtypes = [c_i64]
    lib.pm_fits_stage.argtypes = [c_p, c_p, c_p, c_i, c_p, c_p]
    lib.pm_fits_stage.restype = c_i
    lib.pm_backplanes_map_batch.argtypes = [c_p, c_i, c_p, c_p, c_i64, c_u64, c_p, c_p]
    lib.pm_backplanes_map_batch.restype = c_i
    lib.pm_gather_paired.argtypes = [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_i64, c_i64, c_i, c_u32, c_p, c_p]
    lib.pm_gather_paired.restype = c_i
    lib.pm_gather_grouped.argtypes = [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_i64, c_i64, c_i, c_u32,
                                      c_p, c_p]
    lib.pm_gather_grouped.restype = c_i
    lib.pm_host_ssb_state.argtypes = [c_p, c_i, c_p, c_i, ctypes.c_double, c_p]
    lib.pm_host_ssb_state.restype = c_i
    lib.pm_host_orientation.argtypes = [c_p, ctypes.c_double, c_p, c_p]
    lib.pm_host_orientation.restype = c_i
    for fn in ('pm_backplanes_img', 'pm_backplanes_map', 'pm_backplanes_map_host', 'pm_xy2lonlat', 'pm_lonlat2xy',
               'pm_lonlat2xy_alt',
               'pm_proj_inverse', 'pm_gather', 'pm_spline_prepare', 'pm_fp64_peak_probe',
               'pm_math_probe', 'pm_nan_minmax', 'pm_pchip_resample', 'pm_gather_grid_linear'):
        getattr(lib, fn).restype = c_i
    if lib.pm_abi_version() != 10:
        raise PMLibraryError('libpm_b200.so ABI version mismatch')
    _lib = lib
    return lib


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().pm_error_string(rc).decode()
        raise PMLibraryError(f'{what} failed: {msg} ({rc})')


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise PMLibraryError(
            'planetmapper_b200 needs a CUDA device (sm_100a); there is no CPU fallback'
        )
    return torch


def _stream_ptr(torch) -> int:
    return int(torch.cuda.current_stream().cuda_stream)


def launch_count() -> int:
    return int(load_library().pm_launch_count())


def to_device(arr, device=None):
    torch = _torch()
    import warnings

    a = np.ascontiguousarray(arr, dtype=np.float64)
    with warnings.catch_warnings():
        # read-only views of cached arrays are only ever read (copied to the device) here
        warnings.simplefilter('ignore')
        t = torch.from_numpy(a)
    return t.to(device or 'cuda', non_blocking=False)


# ---- device -> host hand-off ---------------------------------------------------------------
# Results leave the device through PINNED host memory: a pageable destination makes the driver
# stage every copy through its own bounce buffers (about a third of the PCIe rate) and then the
# API's `copy=True` would move the bytes a second time.  The arrays handed to the caller are
# ordinary numpy float64 arrays whose storage is a page-locked block from torch's caching host
# allocator: the block returns to that cache when the array is garbage collected, so a loop that
# drops its results reuses the same blocks and never pays for pinning again.  Page-locked memory is
# a finite resource, so beyond PINNED_BUDGET_BYTES outstanding the copy falls back to pageable memory.
PINNED_BUDGET_BYTES = int(os.environ.get('PM_B200_PINNED_BUDGET', 16 << 30))


def _pinned_outstanding(torch) -> int:
    try:
        return int(torch.cuda.host_memory_stats().get('allocated_bytes.current', 0))
    except Exception:   # older torch: no accounting, no limit
        return 0


def empty_host(shape, torch=None):
    """A float64 CPU tensor for device results: pinned while the budget allows."""
    torch = torch or _torch()
    n = 8
    for d in shape:
        n *= int(d)
    pin = _pinned_outstanding(torch) + n <= PINNED_BUDGET_BYTES
    return torch.empty(tuple(int(d) for d in shape), dtype=torch.float64, pin_memory=pin)


# Staging buffers of the streamed results (Observation.iter_mapped_data): page-locking a gigabyte takes
# about a second, far longer than filling it over PCIe, so ONE set of buffers is kept between calls.
_STAGING = {'buffers': None, 'busy': False}


class staging_buffers:
    """Context manager handing out ``n`` pinned float64 CPU tensors of ``shape``: views of the cached set when
    it is free and large enough, private allocations otherwise (e.g. two streams interleaved)."""

    def __init__(self, shape, n: int = 2):
        self.shape, self.n = tuple(int(d) for d in shape), n
        self.owns_cache = False

    def __enter__(self):
        torch = _torch()
        numel = 1
        for d in self.shape:
            numel *= d
        st = _STAGING
        if not st['busy']:
            bufs = st['buffers']
            if bufs is None or len(bufs) < self.n or bufs[0].numel() < numel:
                st['buffers'] = None     # release the smaller set before pinning the larger one
                bufs = [torch.empty(numel, dtype=torch.float64, pin_memory=True) for _ in range(self.n)]
                st['buffers'] = bufs
            st['busy'] = self.owns_cache = True
            return [b[:numel].view(self.shape) for b in bufs[:self.n]]
        return [torch.empty(self.shape, dtype=torch.float64, pin_memory=True) for _ in range(self.n)]

    def __exit__(self, *exc):
        if self.owns_cache:
            _STAGING['busy'] = False


def release_staging() -> None:
    """Give the cached staging buffers back to the host allocator."""
    if not _STAGING['busy']:
        _STAGING['buffers'] = None


def to_host(dev, out=None):
    """Device tensor -> numpy array (a NEW array the caller owns unless ``out``, a CPU tensor, is given).
    One asynchronous copy on the current stream into pinned memory, then a stream synchronise."""
    torch = _torch()
    host = empty_host(dev.shape, torch) if out is None else out
    host.copy_(dev, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


def popcount(mask: int) -> int:
    return bin(mask & ALL_PLANES).count('1')


def mask_from_names(names) -> int:
    m = 0
    for n in names:
        m |= 1 << PLANE_ID[n]
    return m


def backplanes_img(frames_dev, nx: int, ny: int, mask: int = ALL_PLANES, out=None):
    """frames_dev: CUDA float64 tensor (n_frames, PMFRAME_NDOUBLES). Returns a CUDA
    tensor (n_frames, popcount(mask), ny, nx)."""
    torch = _torch()
    lib = load_library()
    assert frames_dev.is_cuda and frames_dev.dtype == torch.float64 and frames_dev.is_contiguous()
    n_frames = frames_dev.shape[0]
    k = popcount(mask)
    if out is None:
        out = torch.empty((n_frames, k, ny, nx), dtype=torch.float64, device=frames_dev.device)
    rc = lib.pm_backplanes_img(frames_dev.data_ptr(), n_frames, nx, ny, mask, out.data_ptr(),
                               _stream_ptr(torch))
    _check(rc, 'pm_backplanes_img')
    return out


def backplanes_img_host(frame_host, nx: int, ny: int, mask: int = ALL_PLANES, out=None):
    """One frame whose 92 constants are a HOST float64 array: they ride along with the launch as a
    kernel parameter (constant bank).  Returns a CUDA tensor (popcount(mask), ny, nx)."""
    torch = _torch()
    lib = load_library()
    fr = np.ascontiguousarray(frame_host, dtype=np.float64).reshape(-1)
    if fr.size != 92:
        raise ValueError('frame_host must hold the 92 PMFrame doubles')
    if out is None:
        out = torch.empty((popcount(mask), ny, nx), dtype=torch.float64, device='cuda')
    rc = lib.pm_backplanes_img_host(fr.ctypes.data_as(ctypes.c_void_p), nx, ny, mask, out.data_ptr(),
                                    _stream_ptr(torch))
    _check(rc, 'pm_backplanes_img_host')
    return out


def backplanes_map(frame_dev, lon_dev, lat_dev, mask: int = ALL_PLANES, out=None):
    torch = _torch()
    lib = load_library()
    n = lon_dev.numel()
    k = popcount(mask)
    if out is None:
        out = torch.empty((k,) + tuple(lon_dev.shape), dtype=torch.float64, device=lon_dev.device)
    rc = lib.pm_backplanes_map(frame_dev.data_ptr(), lon_dev.data_ptr(), lat_dev.data_ptr(), n,
                               mask, out.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_backplanes_map')
    return out


def backplanes_map_host(frame_host, lon_dev, lat_dev, mask: int = ALL_PLANES, out=None):
    """pm_backplanes_map for one frame whose 92 constants are a HOST float64 array (kernel-parameter
    frame, no upload).  Returns a CUDA tensor (popcount(mask),) + lon_dev.shape."""
    torch = _torch()
    lib = load_library()
    fr = np.ascontiguousarray(frame_host, dtype=np.float64).reshape(-1)
    if fr.size != 92:
        raise ValueError('frame_host must hold the 92 PMFrame doubles')
    assert lon_dev.is_cuda and lat_dev.is_cuda and lon_dev.is_contiguous() and lat_dev.is_contiguous()
    if out is None:
        out = torch.empty((popcount(mask),) + tuple(lon_dev.shape), dtype=torch.float64, device=lon_dev.device)
    rc = lib.pm_backplanes_map_host(fr.ctypes.data_as(ctypes.c_void_p), lon_dev.data_ptr(), lat_dev.data_ptr(),
                                    lon_dev.numel(), mask, out.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_backplanes_map_host')
    return out


def backplanes_points_host(frame_host, x_dev, y_dev, mask: int = ALL_PLANES, *, ring_all: bool = False, out=None):
    """Image-direction planes at arbitrary (fractional, out-of-image) positions ``(x_dev, y_dev)`` of one frame whose
    92 constants are a HOST float64 array (pm_backplanes_points_host).  ``ring_all``: ring-plane coordinates
    without the hidden-behind-the-body test.  Returns a CUDA tensor (popcount(mask),) + x_dev.shape."""
    torch = _torch()
    lib = load_library()
    fr = np.ascontiguousarray(frame_host, dtype=np.float64).reshape(-1)
    if fr.size != 92:
        raise ValueError('frame_host must hold the 92 PMFrame doubles')
    assert x_dev.is_cuda and y_dev.is_cuda and x_dev.is_contiguous() and y_dev.is_contiguous()
    assert x_dev.dtype == torch.float64 and y_dev.dtype == torch.float64 and x_dev.shape == y_dev.shape
    if out is None:
        out = torch.empty((popcount(mask),) + tuple(x_dev.shape), dtype=torch.float64, device=x_dev.device)
    rc = lib.pm_backplanes_points_host(fr.ctypes.data_as(ctypes.c_void_p), x_dev.data_ptr(), y_dev.data_ptr(),
                                       x_dev.numel(), mask, FLAG_RING_ALL if ring_all else 0, out.data_ptr(),
                                       _stream_ptr(torch))
    _check(rc, 'pm_backplanes_points_host')
    return out


def backplanes_map_batch(frames_dev, lon_dev, lat_dev, mask: int = ALL_PLANES, out=None):
    """pm_backplanes_map for every frame of ``frames_dev`` (n_frames, 92) over one lon / lat grid in
    one launch; returns (n_frames, popcount(mask)) + grid shape."""
    torch = _torch()
    lib = load_library()
    assert frames_dev.dim() == 2 and frames_dev.is_contiguous()
    n_frames = frames_dev.shape[0]
    if out is None:
        out = torch.empty((n_frames, popcount(mask)) + tuple(lon_dev.shape), dtype=torch.float64,
                          device=lon_dev.device)
    _check(lib.pm_backplanes_map_batch(frames_dev.data_ptr(), n_frames, lon_dev.data_ptr(), lat_dev.data_ptr(),
                                       lon_dev.numel(), mask, out.data_ptr(), _stream_ptr(torch)),
           'pm_backplanes_map_batch')
    return out


def gather_paired(src, xmaps, ymaps, mode: int, propagate_nan: bool = True, out=None):
    """Plane l of ``src`` mapped with its own maps ``xmaps[l]``, ``ymaps[l]`` (a time series: one image
    and one disc position per frame).  ``src``: CUDA cube (n, ny, nx) for nearest, a :class:`Spline`
    of degree 1 for linear; ``xmaps`` / ``ymaps``: (n,) + map shape, possibly strided along axis 0."""
    torch = _torch()
    lib = load_library()
    spline = src if isinstance(src, Spline) else None
    n, ny, nx = (spline.n_planes, spline.ny, spline.nx) if spline is not None else tuple(src.shape)
    if mode not in (INTERP_NEAREST, INTERP_LINEAR) or (mode == INTERP_LINEAR) != (spline is not None):
        raise ValueError('gather_paired: nearest takes the cube, linear a degree-1 Spline')
    if xmaps.shape != ymaps.shape or xmaps.shape[0] != n or xmaps.stride(0) != ymaps.stride(0):
        raise ValueError('one x / y map per plane, laid out alike')
    n_cells = xmaps[0].numel() if n else 0
    if n and not (xmaps[0].is_contiguous() and ymaps[0].is_contiguous()):
        raise ValueError('each map must be contiguous')
    if out is None:
        out = torch.empty((n,) + tuple(xmaps.shape[1:]), dtype=torch.float64, device=xmaps.device)
    flags = FLAG_PROPAGATE_NAN if propagate_nan else 0
    data = spline.coef if spline is not None else src
    _check(lib.pm_gather_paired(data.data_ptr(), spline.nanbits.data_ptr() if spline is not None else None,
                                spline.plane_bits.data_ptr() if spline is not None else None, n, ny, nx,
                                xmaps.data_ptr(), ymaps.data_ptr(), xmaps.stride(0) if n else n_cells, n_cells, mode,
                                flags, out.data_ptr(), _stream_ptr(torch)), 'pm_gather_paired')
    return out


def gather_grouped(src, xmaps, ymaps, mode: int, planes_per_map: int, plane_stride=None, propagate_nan: bool = True,
                   out=None):
    """Map g of ``xmaps`` / ``ymaps`` ((n_maps,) + map shape, possibly strided along axis 0) applied to the planes
    [g * plane_stride, g * plane_stride + planes_per_map) of ``src`` (a time series of cubes: one cube and one disc
    position per epoch).  ``src``: the CUDA cube (n, ny, nx) for nearest, the :class:`Spline` of the whole cube,
    prepared with ``mode``, for the spline modes.  ``plane_stride`` defaults to ``planes_per_map``.  Returns
    (n_maps, planes_per_map) + map shape."""
    torch = _torch()
    lib = load_library()
    spline = src if isinstance(src, Spline) else None
    if (mode == INTERP_NEAREST) == (spline is not None) or (spline is not None and spline.degree != mode):
        raise ValueError('gather_grouped: nearest takes the cube, a spline mode the Spline prepared with that mode')
    if spline is None and not src.is_contiguous():
        raise ValueError('gather_grouped: the cube must be contiguous')
    n, ny, nx = (spline.n_planes, spline.ny, spline.nx) if spline is not None else tuple(src.shape)
    if xmaps.shape != ymaps.shape or xmaps.stride(0) != ymaps.stride(0):
        raise ValueError('one x / y map per group, laid out alike')
    n_maps = xmaps.shape[0]
    n_cells = xmaps[0].numel() if n_maps else 0
    if n_maps and not (xmaps[0].is_contiguous() and ymaps[0].is_contiguous()):
        raise ValueError('each map must be contiguous')
    plane_stride = planes_per_map if plane_stride is None else plane_stride
    if out is None:
        out = torch.empty((n_maps, planes_per_map) + tuple(xmaps.shape[1:]), dtype=torch.float64, device=xmaps.device)
    flags = FLAG_PROPAGATE_NAN if propagate_nan else 0
    data = spline.coef if spline is not None else src
    _check(lib.pm_gather_grouped(data.data_ptr(), spline.nanbits.data_ptr() if spline is not None else None,
                                 spline.plane_bits.data_ptr() if spline is not None else None, n, ny, nx, n_maps,
                                 planes_per_map, plane_stride, xmaps.data_ptr(), ymaps.data_ptr(),
                                 xmaps.stride(0) if n_maps else n_cells, n_cells, mode, flags, out.data_ptr(),
                                 _stream_ptr(torch)), 'pm_gather_grouped')
    return out


def xy2lonlat(frame_dev, x_dev, y_dev):
    torch = _torch()
    lib = load_library()
    lon = torch.empty_like(x_dev)
    lat = torch.empty_like(x_dev)
    missed = torch.zeros(1, dtype=torch.int64, device=x_dev.device)
    rc = lib.pm_xy2lonlat(frame_dev.data_ptr(), x_dev.data_ptr(), y_dev.data_ptr(),
                          x_dev.numel(), lon.data_ptr(), lat.data_ptr(), missed.data_ptr(),
                          _stream_ptr(torch))
    _check(rc, 'pm_xy2lonlat')
    return lon, lat, missed


def lonlat2xy(frame_dev, lon_dev, lat_dev, not_visible_nan: bool = True, *, alt: float = 0.0,
              planetocentric: bool = False):
    torch = _torch()
    lib = load_library()
    x = torch.empty_like(lon_dev)
    y = torch.empty_like(lon_dev)
    flags = (FLAG_NOT_VISIBLE_NAN if not_visible_nan else 0) | (FLAG_PLANETOCENTRIC if planetocentric else 0)
    rc = lib.pm_lonlat2xy_alt(frame_dev.data_ptr(), lon_dev.data_ptr(), lat_dev.data_ptr(),
                              lon_dev.numel(), float(alt), flags, x.data_ptr(), y.data_ptr(),
                              _stream_ptr(torch))
    _check(rc, 'pm_lonlat2xy_alt')
    return x, y


COORD = {'xy': 0, 'angular': 1, 'km': 2, 'radec': 3, 'lonlat': 4, 'centric': 5}


def transform(frame_dev, src: str, dst: str, a_dev, b_dev, *, alt: float = 0.0, not_visible_nan: bool = False,
              planetocentric: bool = False, aux13=None):
    """Points (a, b) of coordinate system ``src`` in system ``dst`` (pm_transform); returns
    (out_a, out_b, n_missed) as CUDA tensors.  ``aux13``: the obsvec -> angular matrix of the angular system
    (9 doubles, row major) followed by the km -> angular matrix (4), or None for the frame's defaults."""
    torch = _torch()
    lib = load_library()
    oa = torch.empty_like(a_dev)
    ob = torch.empty_like(a_dev)
    missed = torch.zeros(1, dtype=torch.int64, device=a_dev.device)
    flags = (FLAG_NOT_VISIBLE_NAN if not_visible_nan else 0) | (FLAG_PLANETOCENTRIC if planetocentric else 0)
    aux = None
    if aux13 is not None:
        aux = np.ascontiguousarray(aux13, dtype=np.float64).reshape(-1)
        if aux.size != 13:
            raise ValueError('aux13 must hold 9 + 4 doubles')
    rc = lib.pm_transform(frame_dev.data_ptr(), COORD[src], COORD[dst], a_dev.data_ptr(), b_dev.data_ptr(),
                          a_dev.numel(), float(alt), flags,
                          aux.ctypes.data_as(ctypes.c_void_p) if aux is not None else None, oa.data_ptr(),
                          ob.data_ptr(), missed.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_transform')
    return oa, ob, missed


# ---- time series: one launch for the points of every frame (pm_*_batch) --------------------------
MAX_BATCH_FRAMES = 65535   # blockIdx.y of the batched kernels; longer series take one launch per block


def _batch_layout(frames_dev, a_dev, b_dev, per_frame: bool):
    """(n_frames, points per frame, point stride, output shape) of a batched point launch: ``a_dev`` / ``b_dev``
    are contiguous float64 CUDA tensors, (n_frames,) + point shape when ``per_frame``, else the point shape."""
    torch = _torch()
    assert frames_dev.is_cuda and frames_dev.dim() == 2 and frames_dev.shape[1] == 92 and frames_dev.is_contiguous()
    assert a_dev.shape == b_dev.shape and a_dev.is_contiguous() and b_dev.is_contiguous()
    assert a_dev.dtype == torch.float64 and b_dev.dtype == torch.float64
    n_frames = int(frames_dev.shape[0])
    if per_frame:
        if a_dev.dim() < 1 or a_dev.shape[0] != n_frames:
            raise ValueError(f'per-frame points need a leading axis of {n_frames} frames')
        shape = tuple(a_dev.shape[1:])
        n = a_dev[0].numel() if n_frames else 0
        return n_frames, n, n, (n_frames,) + shape
    shape = tuple(a_dev.shape)
    return n_frames, a_dev.numel(), 0, (n_frames,) + shape


def _blocks(n_frames: int):
    for first in range(0, n_frames, MAX_BATCH_FRAMES):
        yield first, min(MAX_BATCH_FRAMES, n_frames - first)


def xy2lonlat_batch(frames_dev, x_dev, y_dev, *, per_frame: bool = False):
    """pm_xy2lonlat_batch: lon / lat (n_frames,) + point shape of every frame of ``frames_dev`` (n_frames, 92), and
    the (n_frames,) int64 counts of missed rays."""
    torch = _torch()
    lib = load_library()
    n_frames, n, stride, shape = _batch_layout(frames_dev, x_dev, y_dev, per_frame)
    lon = torch.empty(shape, dtype=torch.float64, device=frames_dev.device)
    lat = torch.empty_like(lon)
    missed = torch.zeros(n_frames, dtype=torch.int64, device=frames_dev.device)
    for f, m in _blocks(n_frames):
        rc = lib.pm_xy2lonlat_batch(frames_dev[f].data_ptr(), m, x_dev.data_ptr() + 8 * f * stride,
                                    y_dev.data_ptr() + 8 * f * stride, n, stride, lon.data_ptr() + 8 * f * n,
                                    lat.data_ptr() + 8 * f * n, missed[f].data_ptr(), _stream_ptr(torch))
        _check(rc, 'pm_xy2lonlat_batch')
    return lon, lat, missed


def lonlat2xy_batch(frames_dev, lon_dev, lat_dev, *, per_frame: bool = False, not_visible_nan: bool = True,
                    alt: float = 0.0, planetocentric: bool = False):
    """pm_lonlat2xy_batch: x / y (n_frames,) + point shape of every frame of ``frames_dev``."""
    torch = _torch()
    lib = load_library()
    n_frames, n, stride, shape = _batch_layout(frames_dev, lon_dev, lat_dev, per_frame)
    x = torch.empty(shape, dtype=torch.float64, device=frames_dev.device)
    y = torch.empty_like(x)
    flags = (FLAG_NOT_VISIBLE_NAN if not_visible_nan else 0) | (FLAG_PLANETOCENTRIC if planetocentric else 0)
    for f, m in _blocks(n_frames):
        rc = lib.pm_lonlat2xy_batch(frames_dev[f].data_ptr(), m, lon_dev.data_ptr() + 8 * f * stride,
                                    lat_dev.data_ptr() + 8 * f * stride, n, stride, float(alt), flags,
                                    x.data_ptr() + 8 * f * n, y.data_ptr() + 8 * f * n, _stream_ptr(torch))
        _check(rc, 'pm_lonlat2xy_batch')
    return x, y


def transform_batch(frames_dev, src: str, dst: str, a_dev, b_dev, *, per_frame: bool = False, alt: float = 0.0,
                    not_visible_nan: bool = False, planetocentric: bool = False, aux13_dev=None):
    """pm_transform_batch: :func:`transform` for every frame of ``frames_dev``; returns (out_a, out_b) shaped
    (n_frames,) + point shape and the (n_frames,) int64 miss counts.  ``aux13_dev``: (n_frames, 13) CUDA table,
    row f = frame f's ``aux13``, or None for every frame's defaults."""
    torch = _torch()
    lib = load_library()
    n_frames, n, stride, shape = _batch_layout(frames_dev, a_dev, b_dev, per_frame)
    if aux13_dev is not None:
        assert aux13_dev.is_cuda and aux13_dev.dtype == torch.float64 and aux13_dev.is_contiguous()
        if tuple(aux13_dev.shape) != (n_frames, 13):
            raise ValueError(f'aux13 must have shape ({n_frames}, 13)')
    oa = torch.empty(shape, dtype=torch.float64, device=frames_dev.device)
    ob = torch.empty_like(oa)
    missed = torch.zeros(n_frames, dtype=torch.int64, device=frames_dev.device)
    flags = (FLAG_NOT_VISIBLE_NAN if not_visible_nan else 0) | (FLAG_PLANETOCENTRIC if planetocentric else 0)
    for f, m in _blocks(n_frames):
        rc = lib.pm_transform_batch(frames_dev[f].data_ptr(), m, COORD[src], COORD[dst],
                                    a_dev.data_ptr() + 8 * f * stride, b_dev.data_ptr() + 8 * f * stride, n, stride,
                                    float(alt), flags, aux13_dev[f].data_ptr() if aux13_dev is not None else None,
                                    oa.data_ptr() + 8 * f * n, ob.data_ptr() + 8 * f * n, missed[f].data_ptr(),
                                    _stream_ptr(torch))
        _check(rc, 'pm_transform_batch')
    return oa, ob, missed


def proj_inverse(kind: int, a: float, b: float, lon0: float, lat0: float, lon_sign: float,
                 xx_dev, yy_dev):
    torch = _torch()
    lib = load_library()
    params = (ctypes.c_double * 5)(a, b, lon0, lat0, lon_sign)
    lon = torch.empty_like(xx_dev)
    lat = torch.empty_like(xx_dev)
    rc = lib.pm_proj_inverse(kind, ctypes.cast(params, ctypes.c_void_p), xx_dev.data_ptr(),
                             yy_dev.data_ptr(), xx_dev.numel(), lon.data_ptr(), lat.data_ptr(),
                             _stream_ptr(torch))
    _check(rc, 'pm_proj_inverse')
    return lon, lat


def proj_forward(kind: int, a: float, b: float, lon0: float, lat0: float, lon_sign: float, lon_dev, lat_dev):
    torch = _torch()
    lib = load_library()
    params = (ctypes.c_double * 5)(a, b, lon0, lat0, lon_sign)
    xx = torch.empty_like(lon_dev)
    yy = torch.empty_like(lon_dev)
    rc = lib.pm_proj_forward(kind, ctypes.cast(params, ctypes.c_void_p), lon_dev.data_ptr(), lat_dev.data_ptr(),
                             lon_dev.numel(), xx.data_ptr(), yy.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_proj_forward')
    return xx, yy


class Spline:
    """Prepared spline operand of a cube (device buffers filled by pm_spline_prepare;
    layout private to the library, see include/pm_b200.h)."""

    def __init__(self, coef, nanbits, plane_bits, n_planes, ny, nx, degree):
        self.coef, self.nanbits, self.plane_bits = coef, nanbits, plane_bits
        self.n_planes, self.ny, self.nx, self.degree = n_planes, ny, nx, degree

    def planes(self):
        """Coefficients back in the natural (n_planes, ny, nx) layout (tests / debugging)."""
        nq = (self.n_planes + 3) // 4
        c = self.coef.view(nq, self.ny, self.nx, 4).permute(0, 3, 1, 2).reshape(nq * 4, self.ny, self.nx)
        return c[:self.n_planes].contiguous()

    def nanmask(self):
        """Original-NaN mask (n_planes, ny, nx) as a bool tensor (tests / debugging)."""
        import torch

        nw = (self.n_planes + 31) // 32
        w = self.nanbits.view(self.ny, self.nx, nw).to(torch.int64)
        bits = (w[..., None] >> torch.arange(32, device=w.device)) & 1
        return bits.reshape(self.ny, self.nx, nw * 32).permute(2, 0, 1)[:self.n_planes].bool()

    def all_nan_planes(self):
        import torch

        nw = (self.n_planes + 31) // 32
        w = self.plane_bits[:nw].to(torch.int64)
        bits = (w[:, None] >> torch.arange(32, device=w.device)) & 1
        return bits.reshape(-1)[:self.n_planes].bool()


def spline_prepare(cube_dev, degree: int) -> Spline:
    """NaN repair (+ cubic B-spline coefficient solve) packed for :func:`gather`."""
    torch = _torch()
    lib = load_library()
    nl, ny, nx = cube_dev.shape
    dev = cube_dev.device
    coef = torch.empty((lib.pm_spline_coef_bytes(nl, ny, nx) // 8,), dtype=torch.float64, device=dev)
    nanbits = torch.empty((lib.pm_spline_nanbits_bytes(nl, ny, nx) // 4,), dtype=torch.int32, device=dev)
    plane_bits = torch.empty((lib.pm_spline_planebits_bytes(nl) // 4,), dtype=torch.int32, device=dev)
    nbytes = lib.pm_spline_work_bytes(nl, ny, nx, degree)
    work = torch.empty((max(int(nbytes), 256),), dtype=torch.uint8, device=dev)
    rc = lib.pm_spline_prepare(cube_dev.data_ptr(), nl, ny, nx, degree, coef.data_ptr(),
                               nanbits.data_ptr(), plane_bits.data_ptr(), work.data_ptr(),
                               _stream_ptr(torch))
    _check(rc, 'pm_spline_prepare')
    return Spline(coef, nanbits, plane_bits, nl, ny, nx, degree)


def gather(src, xmap_dev, ymap_dev, mode: int, *, plane_begin: int = 0, plane_count=None,
           propagate_nan: bool = True, out=None):
    """Resample planes [plane_begin, plane_begin + plane_count) of a cube onto map cells.
    `src` is the raw CUDA cube (nl, ny, nx) for NEAREST and a :class:`Spline` for
    LINEAR / CUBIC.  Returns (plane_count,) + xmap.shape."""
    torch = _torch()
    lib = load_library()
    if mode == INTERP_NEAREST:
        nl, ny, nx = src.shape
        assert src.is_contiguous()
        ptrs = (src.data_ptr(), None, None)
    else:
        if not isinstance(src, Spline):
            raise PMLibraryError('gather(LINEAR / CUBIC) needs the Spline from spline_prepare()')
        nl, ny, nx = src.n_planes, src.ny, src.nx
        ptrs = (src.coef.data_ptr(), src.nanbits.data_ptr(), src.plane_bits.data_ptr())
    if plane_count is None:
        plane_count = nl - plane_begin
    n_cells = xmap_dev.numel()
    if out is None:
        out = torch.empty((plane_count,) + tuple(xmap_dev.shape), dtype=torch.float64,
                          device=xmap_dev.device)
    flags = FLAG_PROPAGATE_NAN if propagate_nan else 0
    cells_per_row = int(xmap_dev.shape[-1]) if xmap_dev.dim() >= 2 else 0
    rc = lib.pm_gather(ptrs[0], ptrs[1], ptrs[2], nl, ny, nx, plane_begin, plane_count,
                       xmap_dev.data_ptr(), ymap_dev.data_ptr(), n_cells, cells_per_row, mode, flags,
                       out.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_gather')
    return out


class RegridFit:
    """Per-plane smoothing splines of :func:`regrid_fit`: device tensors in fixed-size slots (tx (n, ny +
    k_rows + 1), ty (n, nx + k_cols + 1), c (n, ny * nx), nxy (n, 2) knot counts, fp (n,)), the FITPACK
    ier of every plane as a host array, and the prepared cube (repaired planes, NaN bit planes)."""

    def __init__(self, spline, tx, ty, c, nxy, fp, ier, k_rows, k_cols):
        self.spline, self.tx, self.ty, self.c, self.nxy, self.fp, self.ier = spline, tx, ty, c, nxy, fp, ier
        self.k_rows, self.k_cols = k_rows, k_cols


def regrid_fit(cube_dev, k_rows: int, k_cols: int, s: float, maxit: int = 20) -> RegridFit:
    """RectBivariateSpline(arange(ny), arange(nx), plane, kx=k_rows, ky=k_cols, s=s, maxit=maxit) for every
    plane of a (n, ny, nx) CUDA cube after map_img's NaN repair: one fit launch, then one copy of the ier
    array to the host (the only synchronisation)."""
    torch = _torch()
    lib = load_library()
    nl, ny, nx = cube_dev.shape
    dev = cube_dev.device
    spline = spline_prepare(cube_dev, INTERP_LINEAR)
    tx = torch.empty((nl, ny + k_rows + 1), dtype=torch.float64, device=dev)
    ty = torch.empty((nl, nx + k_cols + 1), dtype=torch.float64, device=dev)
    c = torch.empty((nl, ny * nx), dtype=torch.float64, device=dev)
    nxy = torch.empty((nl, 2), dtype=torch.int32, device=dev)
    fp = torch.empty((nl,), dtype=torch.float64, device=dev)
    ier = torch.empty((nl,), dtype=torch.int32, device=dev)
    nbytes = lib.pm_regrid_work_bytes(nl, ny, nx, k_rows, k_cols)
    if nbytes < 0:
        _check(int(nbytes), 'pm_regrid_work_bytes')
    work = torch.empty((max(int(nbytes), 256),), dtype=torch.uint8, device=dev)
    rc = lib.pm_regrid_fit(spline.coef.data_ptr(), spline.plane_bits.data_ptr(), nl, ny, nx, k_rows, k_cols,
                           float(s), int(maxit), tx.data_ptr(), ty.data_ptr(), c.data_ptr(), nxy.data_ptr(),
                           fp.data_ptr(), ier.data_ptr(), work.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_regrid_fit')
    return RegridFit(spline, tx, ty, c, nxy, fp, ier.cpu().numpy(), k_rows, k_cols)


def gather_regrid(fit: RegridFit, xmap_dev, ymap_dev, *, plane_begin: int = 0, plane_count=None,
                  propagate_nan: bool = True, out=None):
    """Evaluate the splines of planes [plane_begin, plane_begin + plane_count) of :func:`regrid_fit` at the
    map cells (RectBivariateSpline.ev(y, x)).  Returns (plane_count,) + xmap.shape."""
    torch = _torch()
    lib = load_library()
    sp = fit.spline
    if plane_count is None:
        plane_count = sp.n_planes - plane_begin
    if out is None:
        out = torch.empty((plane_count,) + tuple(xmap_dev.shape), dtype=torch.float64, device=xmap_dev.device)
    flags = FLAG_PROPAGATE_NAN if propagate_nan else 0
    rc = lib.pm_gather_regrid(fit.tx.data_ptr(), fit.ty.data_ptr(), fit.c.data_ptr(), fit.nxy.data_ptr(),
                              sp.nanbits.data_ptr(), sp.plane_bits.data_ptr(), sp.n_planes, sp.ny, sp.nx, fit.k_rows,
                              fit.k_cols, plane_begin, plane_count, xmap_dev.data_ptr(), ymap_dev.data_ptr(),
                              xmap_dev.numel(), flags, out.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_gather_regrid')
    return out


def fp64_peak_probe(iters: int = 1 << 15, kind: int = 0) -> float:
    """Measured FP64 FMA throughput in TFLOP/s (8 independent DFMA chains per thread, full grid).
    kind 0: one register operand per DFMA (the datasheet rate); kind 1: three distinct register
    operands per DFMA (what per-pixel vector algebra issues)."""
    _torch()
    lib = load_library()
    ms = ctypes.c_double(0.0)
    fl = ctypes.c_double(0.0)
    _check(lib.pm_fp64_probe(kind, iters, ctypes.byref(ms), ctypes.byref(fl)), 'pm_fp64_probe')
    return fl.value / (ms.value * 1e-3) / 1e12


def math_probe(kind: int, a_dev, b_dev=None):
    """Evaluate one of the library's FP64 primitives elementwise (pm_math_probe)."""
    torch = _torch()
    lib = load_library()
    out = torch.empty_like(a_dev)
    rc = lib.pm_math_probe(kind, a_dev.data_ptr(), b_dev.data_ptr() if b_dev is not None else None,
                           a_dev.numel(), out.data_ptr(), _stream_ptr(torch))
    _check(rc, 'pm_math_probe')
    return out


def nan_minmax(x_dev):
    """(np.nanmin, np.nanmax) of a CUDA tensor, NaN if it holds no finite value."""
    torch = _torch()
    lib = load_library()
    out = torch.empty(2, dtype=torch.float64, device=x_dev.device)
    _check(lib.pm_nan_minmax(x_dev.data_ptr(), x_dev.numel(), out.data_ptr(), _stream_ptr(torch)), 'pm_nan_minmax')
    lo, hi = out.cpu().tolist()
    return lo, hi


def fits_stage(arrays, offsets, image) -> None:
    """Byte-swap the float64 CUDA tensors ``arrays`` into their FITS data units at byte
    ``offsets`` of the uint8 CUDA tensor ``image`` (zero-padded to 2880-byte blocks)."""
    torch = _torch()
    lib = load_library()
    n = len(arrays)
    if n != len(offsets):
        raise ValueError('one offset per array')
    for a in arrays:
        if a.dtype != torch.float64 or not a.is_contiguous() or a.device != image.device:
            raise ValueError('FITS staging needs contiguous float64 tensors on the image device')
    src = (ctypes.c_void_p * n)(*[a.data_ptr() if a.numel() else None for a in arrays])
    cnt = (ctypes.c_int64 * n)(*[a.numel() for a in arrays])
    off = (ctypes.c_int64 * n)(*[int(o) for o in offsets])
    for a, o in zip(arrays, offsets):
        if o + lib.pm_fits_data_unit_bytes(a.numel()) > image.numel():
            raise ValueError('data unit does not fit in the file image')
    _check(lib.pm_fits_stage(src, cnt, off, n, image.data_ptr(), _stream_ptr(torch)), 'pm_fits_stage')


def smooth_grid(n: int, limits, oversample_by: int, max_size: int, limit_padding: float = 5.0):
    """get_xy_pchip of BodyXY._do_smooth_interpolation (body_xy.py:1723-1741): (first original
    index, last original index, number of points of np.linspace(first, last, num))."""
    import math

    first = max(int(math.ceil(limits[0] - limit_padding)), 0)
    last = min(int(math.floor(limits[1] + limit_padding)), n - 1)
    old_size = last - first + 1
    if old_size <= 0:
        return None
    for oversample_to_use in range(int(oversample_by), 1, -1):
        new_size = old_size * oversample_to_use - (oversample_to_use - 1)
        if new_size <= max_size:
            return first, last, new_size
    return first, last, old_size


def map_smooth(cube_dev, xmap_dev, ymap_dev, *, propagate_nan: bool = True, oversample_by: int = 5,
               max_oversampled_img_size: int = 10_000, out=None):
    """BodyXY._do_smooth_interpolation for every plane of a CUDA cube (nl, ny, nx)."""
    torch = _torch()
    lib = load_library()
    nl, ny, nx = cube_dev.shape
    n_cells = xmap_dev.numel()
    if out is None:
        out = torch.empty((nl,) + tuple(xmap_dev.shape), dtype=torch.float64, device=cube_dev.device)
    if n_cells == 0 or nl == 0:
        return out   # a map without cells (xlim / ylim excluded everything)
    xlim, ylim = nan_minmax(xmap_dev), nan_minmax(ymap_dev)
    gx = None if xlim[0] != xlim[0] else smooth_grid(nx, xlim, oversample_by, max_oversampled_img_size)
    gy = None if ylim[0] != ylim[0] else smooth_grid(ny, ylim, oversample_by, max_oversampled_img_size)
    if gx is None or gy is None or gx[2] < 2 or gy[2] < 2:
        out.fill_(float('nan'))   # nothing of the map falls on the image
        return out
    (x0, x1, n_xs), (y0, y1, n_ys) = gx, gy
    fine = torch.empty((nl, n_ys, n_xs), dtype=torch.float64, device=cube_dev.device)
    work = torch.empty((max(int(lib.pm_pchip_work_bytes(nl, ny, nx, n_xs)), 256),), dtype=torch.uint8,
                       device=cube_dev.device)
    _check(lib.pm_pchip_resample(cube_dev.data_ptr(), nl, ny, nx, x0, x1, y0, y1, n_xs, n_ys, fine.data_ptr(),
                                 work.data_ptr(), _stream_ptr(torch)), 'pm_pchip_resample')
    flags = FLAG_PROPAGATE_NAN if propagate_nan else 0
    _check(lib.pm_gather_grid_linear(fine.data_ptr(), nl, n_ys, n_xs, x0, x1, y0, y1, cube_dev.data_ptr(), ny, nx,
                                     xmap_dev.data_ptr(), ymap_dev.data_ptr(), n_cells, flags, out.data_ptr(),
                                     _stream_ptr(torch)), 'pm_gather_grid_linear')
    return out
