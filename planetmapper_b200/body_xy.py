"""
``BodyXY``: the host-side mirror of the reference's ``planetmapper.BodyXY`` for the
accelerated hot path - same method names, argument meaning, return conventions
(float64 host ndarrays, NaN for invalid cells, copies vs read-only cached views)
and cache semantics, with the per-pixel work done by the sm_100a kernels behind
``include/pm_b200.h``.

Reference surface mirrored here (file:line under /root/reference/planetmapper):

- disc parameters            body_xy.py:696-1080 (set/get x0, y0, r0, rotation, img size)
- ``xy2lonlat``/``lonlat2xy`` body_xy.py:433-560
- ``generate_map_coordinates`` body_xy.py:2755-3012
- ``get_backplane_img/map``  body_xy.py:2586-2663, registry :2512-2584, :4198-4356
- ``map_img``                body_xy.py:1414-1631
- caches                     base.py:58-112, body.py:255-272

Design (not the reference's): ONE fused kernel launch produces every image
backplane, so the cache holds one device-resident plane stack per altitude
adjustment instead of one host array per generator; the named getters
(``get_lon_img`` ...) are generated from the backplane table.

Out of scope here, as in SURVEY.md section 8: plotting, wireframes, FITS I/O, disc
fitting, GUI.  Options the kernels do not cover raise ``NotImplementedError``
(there is no CPU fallback).
"""

from __future__ import annotations

import math
from typing import Any, Callable, NamedTuple

import numpy as np

from . import _lib as L
from . import frame as F
from .progress import ProgressMixin, progress_decorator

_PLANE_DESCRIPTIONS = [
    ('LON-GRAPHIC', 'Planetographic longitude, positive {ew} [deg]', 'lon'),
    ('LAT-GRAPHIC', 'Planetographic latitude [deg]', 'lat'),
    ('LON-CENTRIC', 'Planetocentric longitude [deg]', 'lon_centric'),
    ('LAT-CENTRIC', 'Planetocentric latitude [deg]', 'lat_centric'),
    ('RA', 'Right ascension [deg]', 'ra'),
    ('DEC', 'Declination [deg]', 'dec'),
    ('PIXEL-X', 'Observation x pixel coordinate [pixels]', 'x'),
    ('PIXEL-Y', 'Observation y pixel coordinate [pixels]', 'y'),
    ('KM-X', 'East-West distance in target plane [km]', 'km_x'),
    ('KM-Y', 'North-South distance in target plane [km]', 'km_y'),
    ('ANGULAR-X', 'East-West distance in target plane [arcsec]', 'angular_x'),
    ('ANGULAR-Y', 'North-South distance in target plane [arcsec]', 'angular_y'),
    ('PHASE', 'Phase angle [deg]', 'phase_angle'),
    ('INCIDENCE', 'Incidence angle [deg]', 'incidence_angle'),
    ('EMISSION', 'Emission angle [deg]', 'emission_angle'),
    ('AZIMUTH', 'Azimuth angle [deg]', 'azimuth_angle'),
    ('LOCAL-SOLAR-TIME', 'Local solar time [local hours]', 'local_solar_time'),
    ('DISTANCE', 'Distance to observer [km]', 'distance'),
    ('RADIAL-VELOCITY', 'Radial velocity away from observer [km/s]', 'radial_velocity'),
    ('DOPPLER', 'Doppler factor, sqrt((1 + v/c)/(1 - v/c)) where v is radial velocity',
     'doppler'),
    ('LIMB-DISTANCE', 'Distance above limb [km]', 'limb_distance'),
    ('LIMB-LON-GRAPHIC', 'Planetographic longitude of closest point on the limb [deg]',
     'limb_lon'),
    ('LIMB-LAT-GRAPHIC', 'Planetographic latitude of closest point on the limb [deg]',
     'limb_lat'),
    ('RING-RADIUS', 'Equatorial (ring) plane radius [km]', 'ring_plane_radius'),
    ('RING-LON-GRAPHIC', 'Equatorial (ring) plane planetographic longitude [deg]',
     'ring_plane_longitude'),
    ('RING-DISTANCE', 'Equatorial (ring) plane distance to observer [km]',
     'ring_plane_distance'),
]
assert [p[0] for p in _PLANE_DESCRIPTIONS] == L.PLANE_NAMES

_XY_PLANES = (L.PLANE_ID['PIXEL-X'], L.PLANE_ID['PIXEL-Y'])
# the default surface stack (BASELINE config C2): the planes that need the ray / ellipsoid intercept only
_SURFACE_STACK = L.mask_from_names(['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE',
                                    'EMISSION', 'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY',
                                    'DOPPLER'])
_MAP_KWARG_KEYS = ('projection', 'degree_interval', 'lon', 'lat', 'size', 'lon_coords',
                   'lat_coords', 'projection_x_coords', 'projection_y_coords', 'xlim', 'ylim',
                   'alt')


class BackplaneNotFoundError(Exception):
    """Raised when a backplane name is not registered (body_xy.py:2579)."""


class ProjStringError(ValueError):
    """Raised for projection strings this implementation cannot honour."""


class NotFoundError(Exception):
    """Stands in for spiceypy's NotFoundError: a ray missed the target
    (Body._obsvec_norm2lonlat with not_found_nan=False, body.py:1073-1078)."""


def mjd2dtm(mjd: float):
    """Modified Julian Date -> timezone-aware UTC datetime (SpiceBase.mjd2dtm, base.py:500-512; the
    reference goes through astropy.time.Time(mjd, format='mjd').datetime, i.e. the UTC scale with
    MJD 0 = 1858-11-17T00:00:00)."""
    import datetime

    days = math.floor(mjd)
    micro = round((float(mjd) - days) * 86400e6)
    return (datetime.datetime(1858, 11, 17, tzinfo=datetime.timezone.utc)
            + datetime.timedelta(days=days, microseconds=micro))


def standardise_utc_to_string(utc) -> str:
    """BodyBase._standardise_utc_to_string (base.py:841-861): MJD numbers and datetimes (naive ones
    are taken as UTC, aware ones converted to UTC) become '%Y-%m-%dT%H:%M:%S.%f' strings; strings
    pass through."""
    import datetime
    import numbers

    if isinstance(utc, numbers.Number) and not isinstance(utc, bool):
        utc = mjd2dtm(float(utc))
    if isinstance(utc, datetime.datetime):
        if utc.tzinfo is None:
            utc = utc.replace(tzinfo=datetime.timezone.utc)
        utc = utc.astimezone(tz=datetime.timezone.utc).strftime('%Y-%m-%dT%H:%M:%S.%f')
    return str(utc)


class MapTransformer:
    """What ``generate_map_coordinates`` returns in the ``transformer`` slot: the reference hands back the
    ``pyproj.Transformer`` between the body's lon / lat system and the map projection (body_xy.py:3141-3153);
    this object offers the part of its interface the reference and its users call -
    ``transform(xx, yy, direction='FORWARD' | 'INVERSE')`` on scalars or arrays - evaluated by the projection
    kernels (``pm_proj_forward`` / ``pm_proj_inverse``).  FORWARD: planetographic lon / lat (degrees) -> map x / y;
    INVERSE: map x / y -> lon / lat.  Rectangular and manual maps are their own lon / lat system (identity).
    Points a projection cannot show come back as inf, like pyproj's."""

    def __init__(self, kind=None, a=1.0, b=1.0, lon0=0.0, lat0=0.0, lon_sign=1.0, to_kernel=None, from_kernel=None,
                 definition: str = '') -> None:
        self.kind, self.a, self.b, self.lon0, self.lat0, self.lon_sign = kind, a, b, lon0, lat0, lon_sign
        self._to_kernel = to_kernel or (lambda x, y: (x, y))
        self._from_kernel = from_kernel or (lambda x, y: (x, y))
        self.definition = definition

    def __repr__(self) -> str:
        return f'<MapTransformer {self.definition or "lon / lat (identity)"}>'

    def transform(self, xx, yy, direction: str = 'FORWARD'):
        direction = getattr(direction, 'name', str(direction)).upper()
        if direction not in ('FORWARD', 'INVERSE'):
            raise ValueError(f'direction must be FORWARD or INVERSE, not {direction!r}')
        scalar = np.ndim(xx) == 0 and np.ndim(yy) == 0
        a, b = np.broadcast_arrays(np.asarray(xx, dtype=float), np.asarray(yy, dtype=float))
        if self.kind is None:
            u, v = np.array(a), np.array(b)
        elif direction == 'INVERSE':
            xi, yi = self._to_kernel(np.ascontiguousarray(a), np.ascontiguousarray(b))
            lo, la = L.proj_inverse(self.kind, self.a, self.b, self.lon0, self.lat0, self.lon_sign,
                                    L.to_device(xi), L.to_device(yi))
            u, v = L.to_host(lo), L.to_host(la)
        else:
            x, y = L.proj_forward(self.kind, self.a, self.b, self.lon0, self.lat0, self.lon_sign,
                                  L.to_device(np.ascontiguousarray(a)), L.to_device(np.ascontiguousarray(b)))
            u, v = self._from_kernel(L.to_host(x), L.to_host(y))
        if self.kind is not None:
            bad = ~(np.isfinite(u) & np.isfinite(v))
            u = np.where(bad, np.inf, u)
            v = np.where(bad, np.inf, v)
        return (float(u.reshape(())), float(v.reshape(()))) if scalar else (u, v)


class Backplane(NamedTuple):
    """Registry entry, same fields as the reference's Backplane (body_xy.py:79-107)."""

    name: str
    description: str
    get_img: Callable[[], np.ndarray]
    get_map: Callable[..., np.ndarray]


def _readonly(a: np.ndarray) -> np.ndarray:
    v = a.view()
    v.flags.writeable = False
    return v


def _freeze(v: Any):
    """Hashable form of a kwarg value (ndarrays -> nested tuples, base.py:174-199)."""
    if isinstance(v, np.ndarray):
        return ('ndarray', v.shape, tuple(v.ravel().tolist()))
    if isinstance(v, (list, tuple)):
        return tuple(_freeze(x) for x in v)
    return v


# The generated getters live on the instance (and in its `backplanes` registry): they hold the body
# through a weak reference, so that a dropped BodyXY - and the device planes and pinned arrays in its
# caches - is released at once by reference counting instead of waiting for the cycle collector.
def _img_getter(ref, pid: int, stem: str):
    def get_img() -> np.ndarray:
        return ref()._get_img_plane(pid)

    get_img.__name__ = f'get_{stem}_img'
    return get_img


def _map_getter(ref, pid: int, stem: str):
    def get_map(**map_kwargs) -> np.ndarray:
        return ref()._get_map_plane(pid, **map_kwargs)

    get_map.__name__ = f'get_{stem}_map'
    return get_map


_DESCRIPTION_CACHE: dict = {}


def _default_descriptions(ew: str) -> list:
    if ew not in _DESCRIPTION_CACHE:
        _DESCRIPTION_CACHE[ew] = [desc.format(ew=ew) for _, desc, _ in _PLANE_DESCRIPTIONS]
    return _DESCRIPTION_CACHE[ew]


class BodyXY(ProgressMixin):
    """An astronomical body observed at one epoch with an image pixel grid.

    Args mirror ``planetmapper.BodyXY`` (body_xy.py:186-232): ``target``, ``utc``,
    ``observer``, ``nx``, ``ny``, ``sz``.  Extra keyword-only arguments select where
    the once-per-frame constants come from:

    - ``constants``: a prebuilt :class:`planetmapper_b200.frame.BodyConstants`;
    - ``provider``: an ephemeris provider (``spice_host.SpiceProvider`` or
      ``minispice.MiniSpice``); default = :func:`planetmapper_b200.get_default_provider`.
    """

    def __init__(self, target=None, utc=None, observer='EARTH', nx: int = 0, ny: int = 0, *,
                 sz: int | None = None, constants: F.BodyConstants | None = None,
                 provider=None, optimize_speed: bool = True, aberration_correction: str = 'CN',
                 observer_frame: str = 'J2000', target_frame: str | None = None,
                 illumination_source: str = 'SUN',
                 subpoint_method: str = 'INTERCEPT/ELLIPSOID',
                 surface_method: str = 'ELLIPSOID', **kwargs) -> None:
        if kwargs:
            raise TypeError(f'unexpected keyword arguments {sorted(kwargs)}')
        # Scope limits of the kernels (SURVEY.md 8(e)): fail loudly, never fall back.
        if aberration_correction.strip().upper() != 'CN':
            raise NotImplementedError("only aberration_correction='CN' is accelerated")
        if observer_frame.strip().upper() != 'J2000':
            raise NotImplementedError("only observer_frame='J2000' is accelerated")
        if surface_method.strip().upper() != 'ELLIPSOID':
            raise NotImplementedError("only surface_method='ELLIPSOID' is accelerated")
        if illumination_source.strip().upper() != 'SUN':
            raise NotImplementedError("only illumination_source='SUN' is accelerated")
        if subpoint_method.strip().upper() != 'INTERCEPT/ELLIPSOID':
            raise NotImplementedError("only subpoint_method='INTERCEPT/ELLIPSOID' is accelerated")
        if constants is None:
            if provider is None:
                from . import get_default_provider

                provider = get_default_provider()
            if target is None:
                raise TypeError('target is required')
            if utc is None:
                raise NotImplementedError('utc=None (current time) needs a live SPICE setup')
            constants = F.build_body_constants(provider, target, standardise_utc_to_string(utc), observer)
        if target_frame is not None and target_frame.upper() != 'IAU_' + constants.target:
            raise NotImplementedError('only the default IAU_<target> frame is accelerated')
        self._bc = constants
        self._optimize_speed = bool(optimize_speed)
        if sz is not None:
            if nx != 0 or ny != 0:   # body_xy.py:199-201
                raise ValueError('`sz` cannot be used if `nx` and/or `ny` are nonzero')
            nx = ny = sz
        self._nx, self._ny = int(nx), int(ny)
        self._x0 = self._y0 = 0.0
        self._r0 = 10.0
        self._rotation_radians = 0.0
        self._alt_adjustment = 0.0
        self._progress_hook = None
        self._progress_call_stack = []
        self._cache: dict = {}         # cleared when a disc parameter changes
        self._stable_cache: dict = {}  # never cleared
        self.backplanes: dict[str, Backplane] = {}
        self._builtin_getters: dict[str, tuple] = {}
        self._register_default_backplanes()
        # body_xy.py:226-232: centre the disc if an image size was given
        if self._nx > 0 and self._ny > 0:
            self.centre_disc()
        else:
            self._cache['disc method'] = 'default'

    # ---- attributes mirrored from Body (body.py:347-436) ---------------------------
    target = property(lambda self: self._bc.target)
    observer = property(lambda self: self._bc.observer)
    @property
    def dtm(self):
        """Observation time as a timezone-aware datetime (base.py:815-822)."""
        import datetime

        text = str(self._bc.utc).strip().replace(' ', 'T').rstrip('Zz')
        date, _, time = text.partition('T')
        hms = (time.split(':') + ['0', '0', '0'])[:3] if time else ['0', '0', '0']
        sec = float(hms[2] or 0)
        y, mo, d = (int(v) for v in date.split('-'))
        return (datetime.datetime(y, mo, d, int(hms[0] or 0), int(hms[1] or 0), tzinfo=datetime.timezone.utc)
                + datetime.timedelta(seconds=sec))

    # 'YYYY-MM-DDTHH:MM:SS.ffffff', the reference's standardised form of the input time
    utc = property(lambda self: self.dtm.strftime('%Y-%m-%dT%H:%M:%S.%f'))
    et = property(lambda self: self._bc.et)
    target_body_id = property(lambda self: self._bc.target_id)
    radii = property(lambda self: self._bc.radii + self._alt_adjustment)
    r_eq = property(lambda self: float(self._bc.radii[0] + self._alt_adjustment))
    r_polar = property(lambda self: float(self._bc.radii[2] + self._alt_adjustment))
    flattening = property(lambda self: (self.r_eq - self.r_polar) / self.r_eq)
    prograde = property(lambda self: self._bc.prograde)
    positive_longitude_direction = property(lambda self: self._bc.positive_longitude_direction)
    target_light_time = property(lambda self: self._bc.lt0)
    target_distance = property(lambda self: self._bc.target_distance)
    target_ra = property(lambda self: self._bc.target_ra)
    target_dec = property(lambda self: self._bc.target_dec)
    target_diameter_arcsec = property(lambda self: self._bc.target_diameter_arcsec)
    km_per_arcsec = property(lambda self: self._bc.km_per_arcsec)
    subpoint_distance = property(lambda self: self._bc.sub_dist)
    subpoint_lon = property(lambda self: self._bc.subpoint_lon)
    subpoint_lat = property(lambda self: self._bc.subpoint_lat)
    subsol_lon = property(lambda self: self._bc.subsol_lon)
    subsol_lat = property(lambda self: self._bc.subsol_lat)

    def north_pole_angle(self) -> float:
        return self._bc.north_pole_angle

    def speed_of_light(self) -> float:
        return self._bc.clight

    def __repr__(self) -> str:
        return (f'{type(self).__name__}({self.target!r}, {self.utc!r}, observer={self.observer!r}, '
                f'nx={self._nx}, ny={self._ny})')

    # ---- disc parameters (body_xy.py:696-1080) --------------------------------------
    def _clear_cache(self) -> None:
        self._cache.clear()

    def set_x0(self, x0: float) -> None:
        if not math.isfinite(x0):
            raise ValueError('x0 must be finite')
        self._x0 = float(x0)
        self._clear_cache()

    def get_x0(self) -> float:
        return self._x0

    def set_y0(self, y0: float) -> None:
        if not math.isfinite(y0):
            raise ValueError('y0 must be finite')
        self._y0 = float(y0)
        self._clear_cache()

    def get_y0(self) -> float:
        return self._y0

    def set_r0(self, r0: float) -> None:
        if not math.isfinite(r0):
            raise ValueError('r0 must be finite')
        if not r0 > 0:
            raise ValueError('r0 must be greater than zero')
        self._r0 = float(r0)
        self._clear_cache()

    def get_r0(self) -> float:
        return self._r0

    def set_rotation(self, rotation: float) -> None:
        if not math.isfinite(rotation):
            raise ValueError('rotation must be finite')
        self._rotation_radians = float(np.deg2rad(rotation)) % (2 * np.pi)
        self._clear_cache()

    def get_rotation(self) -> float:
        return float(np.rad2deg(self._rotation_radians))

    def set_disc_params(self, x0=None, y0=None, r0=None, rotation=None) -> None:
        if x0 is not None:
            self.set_x0(x0)
        if y0 is not None:
            self.set_y0(y0)
        if r0 is not None:
            self.set_r0(r0)
        if rotation is not None:
            self.set_rotation(rotation)

    def get_disc_params(self) -> tuple[float, float, float, float]:
        return self.get_x0(), self.get_y0(), self.get_r0(), self.get_rotation()

    def set_plate_scale_arcsec(self, arcsec_per_px: float) -> None:
        self.set_r0(self.target_diameter_arcsec / (2 * arcsec_per_px))

    def get_plate_scale_arcsec(self) -> float:
        return self.target_diameter_arcsec / (2 * self.get_r0())

    def get_plate_scale_km(self) -> float:
        return self.get_plate_scale_arcsec() * self.km_per_arcsec

    def set_img_size(self, nx: int | None = None, ny: int | None = None) -> None:
        if nx is not None:
            self._nx = int(nx)
        if ny is not None:
            self._ny = int(ny)
        self._clear_cache()

    def get_img_size(self) -> tuple[int, int]:
        return self._nx, self._ny

    def centre_disc(self) -> None:
        self.set_x0((self._nx - 1) / 2)
        self.set_y0((self._ny - 1) / 2)
        self.set_r0(0.9 * (min(self.get_x0(), self.get_y0())))
        self.set_disc_method('centre_disc')

    def rotate_north_to_top(self) -> None:
        self.set_rotation(-self.north_pole_angle())

    def set_disc_method(self, method: str) -> None:
        self._cache['disc method'] = method

    def get_disc_method(self) -> str:
        return self._cache.get('disc method', 'default')

    # ---- frame handling --------------------------------------------------------------
    def _frame_host(self, alt: float | None = None) -> np.ndarray:
        alt = self._alt_adjustment if alt is None else alt
        return F.pack_frame(self._bc, nx=self._nx, ny=self._ny, x0=self._x0, y0=self._y0,
                            r0=self._r0, rotation_radians=self._rotation_radians, alt=alt,
                            optimize_speed=self._optimize_speed)

    def _frame_dev(self, alt: float | None = None):
        alt = self._alt_adjustment if alt is None else alt
        key = ('frame_dev', alt)
        if key not in self._cache:
            self._cache[key] = L.to_device(self._frame_host(alt))
        return self._cache[key]

    @staticmethod
    def _check_alt(alt: float) -> float:
        alt = float(alt)
        if not math.isfinite(alt):
            raise ValueError('Cannot adjust surface altitude with non-finite alt value')
        return alt

    # ---- point transforms (body_xy.py:433-560, base.py:718-757) ----------------------
    @staticmethod
    def _broadcast(a, b):
        scalar = np.ndim(a) == 0 and np.ndim(b) == 0
        aa, bb = np.broadcast_arrays(np.asarray(a, dtype=float), np.asarray(b, dtype=float))
        return scalar, np.ascontiguousarray(aa), np.ascontiguousarray(bb)

    @staticmethod
    def _unbroadcast(scalar, u, v):
        if scalar:
            return float(u.reshape(())), float(v.reshape(()))
        return u, v

    def xy2lonlat(self, x, y, *, not_found_nan: bool = True, alt: float = 0.0,
                  planetocentric: bool = False):
        """Image pixel coordinates -> planetographic lon/lat (body_xy.py:433-496)."""
        alt = self._check_alt(alt)
        if planetocentric:
            # graphic2centric_lonlat runs INSIDE the altitude adjustment (body.py:1066-1080)
            return self._transform('xy', 'lonlat', x, y, alt=alt, planetocentric=True, not_found_nan=not_found_nan)
        scalar, xa, ya = self._broadcast(x, y)
        fd = self._frame_dev(alt if alt != 0.0 else None)
        lon, lat, missed = L.xy2lonlat(fd, L.to_device(xa), L.to_device(ya))
        lon, lat = L.to_host(lon), L.to_host(lat)
        if not not_found_nan:
            finite_in = np.isfinite(xa) & np.isfinite(ya)
            if int(missed.item()) > 0 or np.any(finite_in & np.isnan(lon)):
                raise NotFoundError('ray does not intercept the target body')
        return self._unbroadcast(scalar, lon, lat)

    def lonlat2xy(self, lon, lat, *, alt: float = 0.0, not_visible_nan: bool = True,
                  planetocentric: bool = False):
        """Planetographic lon/lat -> image pixel coordinates (body_xy.py:498-560)."""
        alt = float(alt)
        scalar, lo, la = self._broadcast(lon, lat)
        if not math.isfinite(alt):   # Body._lonlat2targvec_radians: non-finite alt -> NaN (body.py:900-901)
            return self._unbroadcast(scalar, np.full(lo.shape, np.nan), np.full(lo.shape, np.nan))
        x, y = L.lonlat2xy(self._frame_dev(), L.to_device(lo), L.to_device(la), not_visible_nan,
                           alt=alt, planetocentric=planetocentric)
        return self._unbroadcast(scalar, L.to_host(x), L.to_host(y))

    # ---- the other coordinate pairs (body.py:1083-1900, body_xy.py:385-676) -----------
    def _angular_aux(self, origin_ra=None, origin_dec=None, coordinate_rotation: float = 0.0):
        """Matrices of the angular / km systems for pm_transform (Body._get_obsvec2angular_matrix,
        body.py:1318-1343, with its defaults, and _get_km2angular_matrix, :1625-1634); None when the
        frame's own default matrix applies."""
        if origin_ra is None and origin_dec is None and coordinate_rotation == 0.0:
            return None
        ra = self.target_ra if origin_ra is None else float(origin_ra)
        dec = self.target_dec if origin_dec is None else float(origin_dec)
        m = F.obsvec2angular_matrix(ra, dec, float(coordinate_rotation))
        return np.concatenate([m.ravel(), F.km2angular_matrix(self._bc).ravel()])

    def _transform(self, src: str, dst: str, a, b, *, alt: float = 0.0, not_visible_nan: bool = False,
                   planetocentric: bool = False, not_found_nan: bool = True, angular_kwargs=None):
        """SpiceBase._maybe_transform_as_arrays (base.py:718-757) around one coordinate pair:
        broadcast the two inputs, one kernel launch over all points, floats back if both were scalars."""
        unknown = set(angular_kwargs or ()) - {'origin_ra', 'origin_dec', 'coordinate_rotation'}
        if unknown:
            raise TypeError(f'unexpected angular keyword arguments {sorted(unknown)}')
        alt = float(alt)
        scalar, aa, bb = self._broadcast(a, b)
        if not math.isfinite(alt):
            if dst in ('lonlat', 'centric'):
                self._check_alt(alt)   # _AdjustedSurfaceAltitude raises (body.py:204-207)
            # Body._lonlat2targvec_radians: non-finite alt -> NaN (body.py:900-901)
            return self._unbroadcast(scalar, np.full(aa.shape, np.nan), np.full(aa.shape, np.nan))
        # a lon / lat destination intersects the ellipsoid raised by alt (_AdjustedSurfaceAltitude)
        fd = self._frame_dev(alt if (dst in ('lonlat', 'centric') and src != 'lonlat' and alt != 0.0) else None)
        oa, ob, missed = L.transform(fd, src, dst, L.to_device(aa), L.to_device(bb), alt=alt,
                                     not_visible_nan=not_visible_nan, planetocentric=planetocentric,
                                     aux13=self._angular_aux(**(angular_kwargs or {})))
        if not not_found_nan and int(missed.item()) > 0:
            raise NotFoundError('ray does not intercept the target body')
        return self._unbroadcast(scalar, L.to_host(oa), L.to_host(ob))

    def xy2radec(self, x, y):
        """Image pixel coordinates -> RA / Dec (body_xy.py:385-410)."""
        return self._transform('xy', 'radec', x, y)

    def radec2xy(self, ra, dec):
        """RA / Dec -> image pixel coordinates (body_xy.py:412-437)."""
        return self._transform('radec', 'xy', ra, dec)

    def xy2km(self, x, y):
        """Image pixel coordinates -> km in the target plane (body_xy.py:563-587)."""
        return self._transform('xy', 'km', x, y)

    def km2xy(self, km_x, km_y):
        """km in the target plane -> image pixel coordinates (body_xy.py:589-612)."""
        return self._transform('km', 'xy', km_x, km_y)

    def xy2angular(self, x, y, **angular_kwargs):
        """Image pixel coordinates -> relative angular coordinates, arcsec (body_xy.py:614-645)."""
        return self._transform('xy', 'angular', x, y, angular_kwargs=angular_kwargs)

    def angular2xy(self, angular_x, angular_y, **angular_kwargs):
        """Relative angular coordinates -> image pixel coordinates (body_xy.py:647-676)."""
        return self._transform('angular', 'xy', angular_x, angular_y, angular_kwargs=angular_kwargs)

    def lonlat2radec(self, lon, lat, *, alt: float = 0.0, not_visible_nan: bool = True,
                     planetocentric: bool = False):
        """Body.lonlat2radec (body.py:1083-1146)."""
        return self._transform('lonlat', 'radec', lon, lat, alt=alt, not_visible_nan=not_visible_nan,
                               planetocentric=planetocentric)

    def radec2lonlat(self, ra, dec, *, not_found_nan: bool = True, alt: float = 0.0,
                     planetocentric: bool = False):
        """Body.radec2lonlat (body.py:1148-1221)."""
        return self._transform('radec', 'lonlat', ra, dec, alt=alt, planetocentric=planetocentric,
                               not_found_nan=not_found_nan)

    def radec2angular(self, ra, dec, *, origin_ra=None, origin_dec=None, coordinate_rotation: float = 0.0):
        """Body.radec2angular (body.py:1375-1445)."""
        return self._transform('radec', 'angular', ra, dec, angular_kwargs=dict(
            origin_ra=origin_ra, origin_dec=origin_dec, coordinate_rotation=coordinate_rotation))

    def angular2radec(self, angular_x, angular_y, **angular_kwargs):
        """Body.angular2radec (body.py:1447-1478)."""
        return self._transform('angular', 'radec', angular_x, angular_y, angular_kwargs=angular_kwargs)

    def angular2lonlat(self, angular_x, angular_y, *, not_found_nan: bool = True, alt: float = 0.0,
                       planetocentric: bool = False, **angular_kwargs):
        """Body.angular2lonlat (body.py:1480-1549)."""
        return self._transform('angular', 'lonlat', angular_x, angular_y, alt=alt, planetocentric=planetocentric,
                               not_found_nan=not_found_nan, angular_kwargs=angular_kwargs)

    def lonlat2angular(self, lon, lat, *, alt: float = 0.0, not_visible_nan: bool = True,
                       planetocentric: bool = False, **angular_kwargs):
        """Body.lonlat2angular (body.py:1551-1623)."""
        return self._transform('lonlat', 'angular', lon, lat, alt=alt, not_visible_nan=not_visible_nan,
                               planetocentric=planetocentric, angular_kwargs=angular_kwargs)

    def km2radec(self, km_x, km_y):
        """Body.km2radec (body.py:1652-1675)."""
        return self._transform('km', 'radec', km_x, km_y)

    def radec2km(self, ra, dec):
        """Body.radec2km (body.py:1677-1701)."""
        return self._transform('radec', 'km', ra, dec)

    def km2lonlat(self, km_x, km_y, *, not_found_nan: bool = True, alt: float = 0.0, planetocentric: bool = False):
        """Body.km2lonlat (body.py:1703-1766)."""
        return self._transform('km', 'lonlat', km_x, km_y, alt=alt, planetocentric=planetocentric,
                               not_found_nan=not_found_nan)

    def lonlat2km(self, lon, lat, *, alt: float = 0.0, not_visible_nan: bool = True,
                  planetocentric: bool = False):
        """Body.lonlat2km (body.py:1768-1830)."""
        return self._transform('lonlat', 'km', lon, lat, alt=alt, not_visible_nan=not_visible_nan,
                               planetocentric=planetocentric)

    def km2angular(self, km_x, km_y, **angular_kwargs):
        """Body.km2angular (body.py:1832-1868)."""
        return self._transform('km', 'angular', km_x, km_y, angular_kwargs=angular_kwargs)

    def angular2km(self, angular_x, angular_y, **angular_kwargs):
        """Body.angular2km (body.py:1869-1900)."""
        return self._transform('angular', 'km', angular_x, angular_y, angular_kwargs=angular_kwargs)

    def graphic2centric_lonlat(self, lon, lat, *, alt: float = 0.0):
        """Body.graphic2centric_lonlat (body.py:2915-2947): reclat of pgrrec(lon, lat, alt)."""
        alt = self._check_alt(alt)
        return self._transform('lonlat', 'centric', lon, lat, alt=alt)

    def centric2graphic_lonlat(self, lon_centric, lat_centric, *, alt: float = 0.0):
        """Body.centric2graphic_lonlat (body.py:2949-2982): latsrf, then recpgr against the spheroid raised
        by alt."""
        alt = self._check_alt(alt)
        return self._transform('lonlat', 'lonlat', lon_centric, lat_centric, alt=alt, planetocentric=True)

    # ---- per-point geometry (body.py:2081-2110, :2152-2615) ------------------------------
    # Vectorised forms of the reference's scalar queries: scalars give floats, arrays give float64
    # arrays of the broadcast shape, and each call is a fixed number of launches whatever the number of
    # points.  Nothing here is cached (the reference caches none of them) and no image size is needed.
    @staticmethod
    def _refuse_point_alt(alt) -> None:
        if float(alt) != 0.0:
            # the reference's meaning of a point above the ellipsoid (illumf's normal, spkcpt at an
            # off-surface point) is not pinned by any test here: refuse rather than guess
            raise NotImplementedError('alt != 0 is not supported by the lon / lat point methods')

    def _lonlat_point_planes(self, lon, lat, names):
        """The map-direction planes ``names`` at the cells (lon, lat): one pm_backplanes_map_host launch, the
        values get_backplane_map gives for those cells."""
        scalar, lo, la = self._broadcast(lon, lat)
        mask = L.mask_from_names(names)
        planes = L.to_host(L.backplanes_map_host(self._frame_host(), L.to_device(lo), L.to_device(la), mask))
        return scalar, [planes[L.popcount(mask & ((1 << L.PLANE_ID[n]) - 1))] for n in names]

    def _radec_point_planes(self, ra, dec, names, *, ring_all: bool = False):
        """The image-direction planes ``names`` along the directions (ra, dec): pm_transform radec -> xy, then
        pm_backplanes_points_host at those (fractional) pixel positions - two launches."""
        scalar, a, b = self._broadcast(ra, dec)
        mask = L.mask_from_names(names)
        x, y, _ = L.transform(self._frame_dev(), 'radec', 'xy', L.to_device(a), L.to_device(b))
        planes = L.to_host(L.backplanes_points_host(self._frame_host(), x, y, mask, ring_all=ring_all))
        return scalar, [planes[L.popcount(mask & ((1 << L.PLANE_ID[n]) - 1))] for n in names]

    @staticmethod
    def _point_result(scalar, arrays):
        if scalar:
            values = tuple(float(a.reshape(())) for a in arrays)
        else:
            values = tuple(arrays)
        return values if len(values) > 1 else values[0]

    def illumination_angles_from_lonlat(self, lon, lat, *, alt: float = 0.0):
        """Body.illumination_angles_from_lonlat: (phase, incidence, emission) in degrees at a surface point;
        angles of points on the far side are returned too (emission > 90)."""
        self._refuse_point_alt(alt)
        scalar, planes = self._lonlat_point_planes(lon, lat, ['PHASE', 'INCIDENCE', 'EMISSION'])
        return self._point_result(scalar, planes)

    def azimuth_angle_from_lonlat(self, lon, lat, *, alt: float = 0.0):
        """Body.azimuth_angle_from_lonlat: azimuth angle in degrees at a surface point."""
        self._refuse_point_alt(alt)
        scalar, planes = self._lonlat_point_planes(lon, lat, ['AZIMUTH'])
        return self._point_result(scalar, planes)

    def local_solar_time_from_lon(self, lon):
        """Body.local_solar_time_from_lon: local solar time in decimal local hours (et2lst's whole seconds)."""
        scalar, planes = self._lonlat_point_planes(lon, 0.0, ['LOCAL-SOLAR-TIME'])
        return self._point_result(scalar, planes)

    @staticmethod
    def _lst_string(hours) -> str:
        if not math.isfinite(hours):
            return 'nan'
        total = round(hours * 3600)   # the decimal hours are h + m / 60 + s / 3600 of et2lst's integers
        return '%02d:%02d:%02d' % (total // 3600, (total % 3600) // 60, total % 60)

    def local_solar_time_string_from_lon(self, lon):
        """Body.local_solar_time_string_from_lon: local solar time as 'HH:MM:SS' (an array of '<U8' strings for
        array input; 'nan' where lon is not finite)."""
        hours = self.local_solar_time_from_lon(lon)
        if np.ndim(hours) == 0:
            return self._lst_string(float(hours))
        out = np.empty(np.shape(hours), dtype='<U8')
        flat = out.reshape(-1)
        for i, h in enumerate(np.asarray(hours).reshape(-1).tolist()):
            flat[i] = self._lst_string(h)
        return out

    def distance_from_lonlat(self, lon, lat, *, alt: float = 0.0):
        """Body.distance_from_lonlat: distance from the observer to a surface point, km."""
        self._refuse_point_alt(alt)
        scalar, planes = self._lonlat_point_planes(lon, lat, ['DISTANCE'])
        return self._point_result(scalar, planes)

    def radial_velocity_from_lonlat(self, lon, lat, *, alt: float = 0.0):
        """Body.radial_velocity_from_lonlat: radial velocity of a surface point away from the observer, km/s."""
        self._refuse_point_alt(alt)
        scalar, planes = self._lonlat_point_planes(lon, lat, ['RADIAL-VELOCITY'])
        return self._point_result(scalar, planes)

    def test_if_lonlat_visible(self, lon, lat, alt: float = 0.0):
        """Body.test_if_lonlat_visible: True where the point (at altitude ``alt`` above the surface) faces the
        observer and nothing of the body hides it; a bool array for array input."""
        ra, dec = self.lonlat2radec(lon, lat, alt=alt, not_visible_nan=True)
        visible = np.isfinite(ra) & np.isfinite(dec)
        return bool(visible) if np.ndim(visible) == 0 else visible

    def limb_coordinates_from_radec(self, ra, dec):
        """Body.limb_coordinates_from_radec: (lon, lat, distance) of the limb point nearest to the direction
        (ra, dec); distance is km above the limb (negative inside the disc)."""
        scalar, planes = self._radec_point_planes(ra, dec, ['LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC', 'LIMB-DISTANCE'])
        return self._point_result(scalar, planes)

    def ring_plane_coordinates(self, ra, dec, only_visible: bool = True):
        """Body.ring_plane_coordinates: (radius km, planetographic longitude deg, distance km) where the direction
        (ra, dec) meets the equatorial (ring) plane; NaN where it does not, and with ``only_visible`` also where
        the body hides that point."""
        scalar, planes = self._radec_point_planes(ra, dec, ['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE'],
                                                  ring_all=not only_visible)
        return self._point_result(scalar, planes)

    # ---- projections (body_xy.py:2755-3012) -------------------------------------------
    def generate_map_coordinates(self, projection: str = 'rectangular', *,
                                 degree_interval: float = 1, lon: float = 0, lat: float = 0,
                                 size: int = 100, lon_coords=None, lat_coords=None,
                                 projection_x_coords=None, projection_y_coords=None,
                                 xlim=None, ylim=None, alt: float = 0.0):
        """Returns ``(lons, lats, xx, yy, transformer, info)`` like the reference; ``transformer`` is a
        :class:`MapTransformer` (the ``transform(xx, yy, direction=...)`` part of pyproj's interface on the
        projection kernels)."""
        info: dict[str, Any]
        transformer = MapTransformer()     # rectangular / manual: the map is the lon / lat system itself
        a, b = self._bc.r_eq + alt, self._bc.r_polar + alt
        lon_sign = self._bc.lon_sign
        if projection == 'rectangular':
            lons = np.arange(degree_interval / 2, 360, degree_interval)
            if self.positive_longitude_direction == 'W':
                lons = lons[::-1]
            lats = np.arange(-90 + degree_interval / 2, 90, degree_interval)
            lons, lats = np.meshgrid(lons.astype(float, copy=False), lats.astype(float, copy=False))
            xx, yy = lons, lats
            info = dict(projection=projection, degree_interval=degree_interval)
        elif projection == 'manual':
            if lon_coords is None or lat_coords is None:
                raise ValueError(
                    'lon_coords and lat_coords must be provided for manual projection')
            lons = np.asarray(lon_coords)
            lats = np.asarray(lat_coords)
            if lons.ndim != lats.ndim:
                raise ValueError(
                    'lon_coords and lat_coords must have the same number of dimensions')
            if lons.ndim == 1:
                lons, lats = np.meshgrid(lons, lats)
            if lons.ndim != 2:
                raise ValueError('lon_coords and lat_coords must be 1D or 2D arrays')
            if lons.shape != lats.shape:
                raise ValueError('lon_coords and lat_coords must have the same shape')
            lons = np.array(lons, dtype=float)
            lats = np.array(lats, dtype=float)
            xx, yy = lons, lats
            info = dict(projection=projection)
        elif projection in ('orthographic', 'azimuthal', 'azimuthal equal area'):
            if projection == 'orthographic':
                kind, lim = L.PROJ_ORTHOGRAPHIC, max(1, b / a) * 1.01
            elif projection == 'azimuthal':
                kind, lim = L.PROJ_AZIMUTHAL, 1.01
            else:
                kind, lim = L.PROJ_AZIMUTHAL_EQUAL_AREA, 1.01
            c = np.linspace(-lim, lim, size)
            xx, yy = np.meshgrid(c, c)
            lo, la = L.proj_inverse(kind, a, b, float(lon), float(lat), lon_sign,
                                    L.to_device(xx), L.to_device(yy))
            lons, lats = L.to_host(lo), L.to_host(la)
            transformer = MapTransformer(kind, a, b, float(lon), float(lat), lon_sign,
                                         definition=f'{projection} lon_0={lon} lat_0={lat} a={a} b={b}')
            info = dict(projection=projection, lon=lon, lat=lat, size=size)
        else:
            # custom proj string (body_xy.py:2970-2980)
            if projection_x_coords is None:
                raise ValueError('x coords must be provided')
            lons, lats, xx, yy, transformer = self._custom_proj_map_coords(projection, projection_x_coords,
                                                                          projection_y_coords)
            info = dict(projection=projection, projection_x_coords=projection_x_coords,
                        projection_y_coords=projection_y_coords)
        info['xlim'] = xlim
        info['ylim'] = ylim
        if xlim is not None:
            x_arr = xx[0]
            keep = (x_arr >= min(xlim)) & (x_arr <= max(xlim))
            xx, yy, lons, lats = xx[:, keep], yy[:, keep], lons[:, keep], lats[:, keep]
        if ylim is not None:
            y_arr = yy[:, 0]
            keep = (y_arr >= min(ylim)) & (y_arr <= max(ylim))
            xx, yy, lons, lats = xx[keep, :], yy[keep, :], lons[keep, :], lats[keep, :]
        same = xx is lons
        # every branch above built fresh arrays; inf -> NaN (body_xy.py:3005-3006) only where there is one
        lons = np.asarray(lons, dtype=float)
        lats = np.asarray(lats, dtype=float)
        if not np.isfinite(lons).all():
            lons = np.where(np.isfinite(lons), lons, np.nan)
        if not np.isfinite(lats).all():
            lats = np.where(np.isfinite(lats), lats, np.nan)
        if same:
            xx, yy = lons, lats
        if alt != 0.0:
            info['alt'] = alt
        return _readonly(lons), _readonly(lats), _readonly(xx), _readonly(yy), transformer, info

    def create_proj_string(self, proj: str, **parameters) -> str:
        """Proj string with this body's radii and axis direction filled in
        (body_xy.py:3056-3095): ``a``, ``b`` and ``axis`` default to the body's values and a
        parameter given as ``None`` is left out."""
        merged = dict(parameters)
        merged.setdefault('a', self.r_eq)
        merged.setdefault('b', self.r_polar)
        merged.setdefault('axis', f'{self.positive_longitude_direction.lower()}nu')
        parts = [f'+proj={proj}'] + [f'+{k}={v}' for k, v in merged.items() if v is not None]
        return ' '.join(parts + ['+type=crs'])

    def _check_proj_string_for_axis(self, projection: str) -> None:
        expected_axis = f'+axis={self.positive_longitude_direction.lower()}nu'   # body_xy.py:3097-3104
        if expected_axis not in projection:
            raise ProjStringError(
                f'Projection string {projection!r} does not have the expected axis orientation '
                f'{expected_axis!r} for positive {self.positive_longitude_direction} coordinates.')

    # proj parameters the device kernels cover (pm_proj_inverse): ortho on an ellipsoid, aeqd /
    # laea on a sphere, with the linear +to_meter / +x_0 / +y_0 terms folded into the grid
    _PROJ_KINDS = {'ortho': L.PROJ_ORTHOGRAPHIC, 'aeqd': L.PROJ_AZIMUTHAL, 'laea': L.PROJ_AZIMUTHAL_EQUAL_AREA}

    def _custom_proj_map_coords(self, projection: str, xx, yy):
        """``_get_pyproj_map_coords`` (body_xy.py:3106-3128) for the proj strings whose inverse the
        CUDA kernels implement; anything else raises ProjStringError (there is no PROJ here)."""
        if yy is None:
            yy = xx
        xx, yy = np.asarray(xx), np.asarray(yy)
        if xx.ndim != yy.ndim:
            raise ValueError('x and y coords must have the same number of dimensions')
        if xx.ndim == 1:
            xx, yy = np.meshgrid(xx, yy)
        if xx.ndim != 2:
            raise ValueError('x and y coords must be 1D or 2D arrays')
        if xx.shape != yy.shape:
            raise ValueError('x and y coords must have the same shape')
        self._check_proj_string_for_axis(projection)
        par: dict[str, str | None] = {}
        for token in projection.split():
            key, sep, value = token.lstrip('+').partition('=')
            par[key] = value if sep else None
        known = {'proj', 'R', 'a', 'b', 'lon_0', 'lat_0', 'x_0', 'y_0', 'to_meter', 'axis', 'type', 'units',
                 'no_defs'}
        unknown = sorted(set(par) - known)
        kind = self._PROJ_KINDS.get(par.get('proj') or '')
        if kind is None or unknown or par.get('units') not in (None, 'm'):
            raise ProjStringError(
                f'proj string {projection!r} is outside the accelerated subset: +proj=ortho|aeqd|laea with '
                f'+R | +a +b, +lon_0, +lat_0, +x_0, +y_0, +to_meter, +axis (unsupported: '
                f'{unknown or par.get("proj") or par.get("units")})')

        def num(key: str, default: float) -> float:
            v = par.get(key)
            try:
                return default if v is None else float(v)
            except ValueError as exc:
                raise ProjStringError(f'bad value for +{key} in {projection!r}') from exc

        if 'R' in par:
            a = b = num('R', 1.0)
        elif 'a' in par:
            a = num('a', 1.0)
            b = num('b', a) if 'b' in par else a   # PROJ: +a without a second shape parameter is a sphere
        else:
            # PROJ would silently fall back to the GRS80 Earth ellipsoid here
            raise ProjStringError(f'{projection!r} needs an explicit +R or +a (create_proj_string adds them)')
        if not (a > 0 and b > 0):
            raise ProjStringError(f'radii must be positive in {projection!r}')
        if kind != L.PROJ_ORTHOGRAPHIC and a != b:
            raise ProjStringError(f'+proj={par["proj"]} is only accelerated on a sphere (+R or +a without +b)')
        lon0, lat0 = num('lon_0', 0.0), num('lat_0', 0.0)
        tm = num('to_meter', 1.0)
        # PROJ inverse: internal = (user * to_meter - false origin) / a; then the units the
        # kernels take (the reference's own strings: to_meter = a, a pi and 2 a; y_0 of the ortho)
        x_0, y_0 = num('x_0', 0.0), num('y_0', 0.0)
        y_shift = (b / a - 1.0) * np.sin(np.radians(lat0 * 2)) if kind == L.PROJ_ORTHOGRAPHIC else 0.0
        unit = {L.PROJ_ORTHOGRAPHIC: 1.0, L.PROJ_AZIMUTHAL: np.pi, L.PROJ_AZIMUTHAL_EQUAL_AREA: 2.0}[kind]

        def to_kernel(x, y):      # the caller's units -> the kernels' (the reference's own strings: to_meter = a, a pi, 2 a)
            return ((np.asarray(x, dtype=float) * tm - x_0) / a / unit,
                    ((np.asarray(y, dtype=float) * tm - y_0) / a + y_shift) / unit)

        def from_kernel(x, y):
            return (x * unit * a + x_0) / tm, ((y * unit - y_shift) * a + y_0) / tm

        transformer = MapTransformer(kind, a, b, lon0, lat0, self._bc.lon_sign, to_kernel, from_kernel, projection)
        xi, yi = to_kernel(xx, yy)
        lo, la = L.proj_inverse(kind, a, b, lon0, lat0, self._bc.lon_sign, L.to_device(xi), L.to_device(yi))
        return L.to_host(lo), L.to_host(la), xx, yy, transformer

    # ---- backplane registry (body_xy.py:2512-2584) -------------------------------------
    @staticmethod
    def standardise_backplane_name(name: str) -> str:
        return name.strip().upper()

    def register_backplane(self, name, description, get_img, get_map) -> None:
        name = self.standardise_backplane_name(name)
        if name in self.backplanes:
            raise ValueError(f'Backplane named {name!r} is already registered')
        self.backplanes[name] = Backplane(name, description, get_img, get_map)

    def get_backplane(self, name: str) -> Backplane:
        name = self.standardise_backplane_name(name)
        try:
            return self.backplanes[name]
        except KeyError as exc:
            raise BackplaneNotFoundError(
                '{n!r} not found. Currently registered backplanes are: {r}.'.format(
                    n=name, r=', '.join(repr(n) for n in self.backplanes))) from exc

    def backplane_summary_string(self) -> str:
        return '\n'.join(f'{bp.name}: {bp.description}' for bp in self.backplanes.values())

    def _register_default_backplanes(self) -> None:
        # one pass over the 26 defaults (body_xy.py:4198-4356); this runs in every constructor, i.e. inside every
        # end-to-end step, so it avoids per-plane method calls: 52 closures over ONE weak reference
        import weakref

        ew = self.positive_longitude_direction  # body_xy.py:4201-4203
        descriptions = _default_descriptions(ew)
        ref = weakref.ref(self)
        attrs, backplanes, builtin = self.__dict__, self.backplanes, self._builtin_getters
        for pid, (name, _, stem) in enumerate(_PLANE_DESCRIPTIONS):
            get_img = _img_getter(ref, pid, stem)
            get_map = _map_getter(ref, pid, stem)
            attrs[f'get_{stem}_img'] = get_img
            attrs[f'get_{stem}_map'] = get_map
            backplanes[name] = Backplane(name, descriptions[pid], get_img, get_map)
            builtin[name] = (get_img, get_map)

    def _is_builtin_backplane(self, name: str, mapped: bool) -> bool:
        """True while ``backplanes[name]`` is still the kernel-backed default getter."""
        getters = self._builtin_getters.get(name)
        bp = self.backplanes.get(name)
        if getters is None or bp is None:
            return False
        return (bp.get_map is getters[1]) if mapped else (bp.get_img is getters[0])

    # ---- image-direction backplanes ----------------------------------------------------
    def _test_if_img_size_valid(self) -> bool:
        return (self._nx > 0) and (self._ny > 0)

    @progress_decorator
    def get_backplanes_img_device(self, mask: int = L.ALL_PLANES, alt: float | None = None):
        """All requested image backplanes as ONE device tensor (k, ny, nx), computed by a
        single fused kernel launch and cached per altitude adjustment in ``_cache``
        (cleared with the disc parameters, like the reference's
        ``_cache_clearable_alt_dependent_result``, body.py:255-272)."""
        if not self._test_if_img_size_valid():
            raise ValueError('nx and ny must be positive to create a backplane image')
        alt = self._alt_adjustment if alt is None else alt
        key = ('img_planes_dev', alt)
        entry = self._cache.get(key)
        if entry is None or (entry[0] & mask) != mask:
            have = entry[0] if entry else 0
            new_mask = have | mask
            if (new_mask & ~_SURFACE_STACK) == 0:
                # surface planes share the ray / ellipsoid intercept, which is nearly all of their cost: one
                # plane or the 12-plane stack (specialised kernel, 0.15 ms for 2048 x 2048) are the same work
                new_mask = _SURFACE_STACK
            elif have:
                # second distinct request outside the surface stack: everything (at most two launches for any
                # sequence of single-plane getters, and a lone RA / ring plane never pays for the 26-plane stack)
                new_mask = L.ALL_PLANES
            # single frame: the constants ride in the launch (kernel parameter / constant bank)
            planes = L.backplanes_img_host(self._frame_host(alt), self._nx, self._ny, new_mask)
            entry = (new_mask, planes)
            self._cache[key] = entry   # host copies already handed out stay valid (same values)
        return entry

    def _get_img_plane(self, pid: int) -> np.ndarray:
        alt = self._alt_adjustment
        key = ('img_host', pid, alt)
        if key not in self._cache:
            # only the requested plane is added to what the cache already holds (a single
            # get_backplane_img('EMISSION') must not pay for the 26-plane stack)
            have, planes = self.get_backplanes_img_device(1 << pid, alt)
            slot = L.popcount(have & ((1 << pid) - 1))
            self._cache[key] = _readonly(L.to_host(planes[slot]))
        return self._cache[key]

    def get_backplane_img(self, name: str, *, alt: float = 0.0) -> np.ndarray:
        """Copy of a backplane image (body_xy.py:2586-2630)."""
        alt = self._check_alt(alt)
        bp = self.get_backplane_or_keyerror(name)
        with _AltitudeScope(self, alt):
            if self._is_builtin_backplane(bp.name, mapped=False):
                # the cache is the device-resident plane stack: ONE copy, device -> the (pinned) array the
                # caller gets, instead of device -> cached host array -> np.array(copy=True)
                return self._img_plane_to_host(L.PLANE_ID[bp.name])
            return np.array(bp.get_img(), copy=True)

    # Planes at least this large are read ahead (below it the per-call overhead is not the copy)
    _PREFETCH_MIN_BYTES = 4 << 20
    # Planes kept in flight ahead of the caller: enough to bridge Python's return to the caller and its next
    # request (a copy of a 2048 x 2048 plane takes 0.6 ms), few enough that a caller who wanted ONE plane has
    # paid for two small background copies, not for the whole stack
    _PREFETCH_WINDOW = 2

    def _img_plane_to_host(self, pid: int) -> np.ndarray:
        """A new host array holding image plane ``pid``.  The usual caller asks for one backplane after the
        other (the reference's save_observation loop, observation.py:1275, or user code), so the copy engine is
        kept busy across the calls: the requested plane is copied device -> pinned host on a side stream and,
        BEFORE waiting for it, the next ``_PREFETCH_WINDOW`` planes of the stack nobody has asked for yet are
        queued behind it.  Each read-ahead array is handed to the first request for its plane (ownership moves
        to the caller); later requests copy again."""
        torch = L._torch()
        alt = self._alt_adjustment
        have, planes = self.get_backplanes_img_device(1 << pid, alt)
        slot = lambda q: L.popcount(have & ((1 << q) - 1))   # noqa: E731
        if planes[0].numel() * 8 < self._PREFETCH_MIN_BYTES:
            return L.to_host(planes[slot(pid)])
        key = ('img_readahead', alt)
        state = self._cache.get(key)
        if state is None or state['planes'] is not planes:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())    # the kernel that fills `planes`
            planes.record_stream(side)     # the stack must outlive the copies even if the cache is cleared meanwhile
            state = {'planes': planes, 'asked': set(), 'ready': {}, 'stream': side}
            self._cache[key] = state
        side = state['stream']

        def enqueue(q):
            host = L.empty_host(planes[slot(q)].shape, torch)
            if not host.is_pinned():
                return None            # pinned budget exhausted: no asynchronous copy into pageable memory
            host.copy_(planes[slot(q)], non_blocking=True)
            event = torch.cuda.Event()
            event.record(side)
            return host, event

        mine = state['ready'].pop(pid, None)
        state['asked'].add(pid)
        with torch.cuda.stream(side):
            if mine is None:
                mine = enqueue(pid)
            if mine is not None:
                ahead = len(state['ready'])
                for q in range(L.N_PLANES):
                    if ahead >= self._PREFETCH_WINDOW:
                        break
                    if (have >> q) & 1 and q not in state['asked'] and q not in state['ready']:
                        nxt = enqueue(q)
                        if nxt is None:
                            break
                        state['ready'][q] = nxt
                        ahead += 1
        if mine is None:
            return L.to_host(planes[slot(pid)])
        host, event = mine
        event.synchronize()
        return host.numpy()

    def get_backplane_imgs(self, names, *, alt: float = 0.0, out=None) -> dict[str, np.ndarray]:
        """Several backplane images from ONE kernel launch and ONE device->host copy.

        Equivalent to ``{n: body.get_backplane_img(n, alt=alt) for n in names}`` but only
        the requested planes are computed and they cross PCIe together.  ``out`` may be a
        pinned CPU tensor of shape (len(names), ny, nx) to receive the data (the returned
        arrays are then views of it); otherwise fresh host memory is allocated.
        """
        torch = L._torch()
        alt = self._check_alt(alt)
        std = [self.standardise_backplane_name(n) for n in names]
        for n in std:
            if n not in L.PLANE_ID:
                raise BackplaneNotFoundError(f'{n!r} is not a built-in backplane')
        if not self._test_if_img_size_valid():
            raise ValueError('nx and ny must be positive to create a backplane image')
        mask = L.mask_from_names(std)
        planes = L.backplanes_img_host(self._frame_host(alt), self._nx, self._ny, mask)
        order = sorted(set(std), key=lambda n: L.PLANE_ID[n])
        if out is None:
            host = L.empty_host(planes.shape)
            host.copy_(planes, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        else:
            host = out[: len(order)]
            host.copy_(planes, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        arr = host.numpy()
        return {n: arr[order.index(n)] for n in std}

    def get_backplane_or_keyerror(self, name: str) -> Backplane:
        # the reference indexes the dict directly here (KeyError), body_xy.py:2627
        return self.backplanes[self.standardise_backplane_name(name)]

    # ---- map-direction backplanes ------------------------------------------------------
    def _map_key(self, map_kwargs: dict) -> tuple:
        unknown = set(map_kwargs) - set(_MAP_KWARG_KEYS)
        if unknown:
            raise TypeError(f'unexpected map keyword arguments {sorted(unknown)}')
        return tuple(sorted((k, _freeze(v)) for k, v in map_kwargs.items()))

    def _get_lonlat_planes(self, **map_kwargs) -> tuple[np.ndarray, np.ndarray]:
        """lon % 360 and lat of every map cell (body_xy.py:3293-3300) as two contiguous planes - the layout
        the kernels take; stable cache."""
        key = ('lonlat_planes', self._map_key(map_kwargs))
        if key not in self._stable_cache:
            lons, lats, *_ = self.generate_map_coordinates(**map_kwargs)
            if lons.size and not (np.nanmin(lons) >= 0.0 and np.nanmax(lons) < 360.0):
                lons = lons % 360       # already in [0, 360) for the built-in grids: skip the pass
            self._stable_cache[key] = (_readonly(np.ascontiguousarray(lons)), _readonly(np.ascontiguousarray(lats)))
        return self._stable_cache[key]

    def _get_lonlat_map(self, **map_kwargs) -> np.ndarray:
        """(n0, n1, 2) lon % 360, lat, the reference's layout (body_xy.py:3293-3300)."""
        lons, lats = self._get_lonlat_planes(**map_kwargs)
        return _readonly(np.stack([lons, lats], axis=-1))

    @progress_decorator
    def get_backplanes_map_device(self, mask: int, **map_kwargs):
        """Requested map backplanes as a device tensor (k, n0, n1).  Disc-independent
        planes live in ``_stable_cache`` (never cleared), PIXEL-X / PIXEL-Y (x_map,
        y_map) in ``_cache`` - the reference's split (body_xy.py:3423 vs :3482)."""
        alt = self._check_alt(map_kwargs.get('alt', 0.0))
        mkey = self._map_key(map_kwargs)
        xy_mask = mask & ((1 << _XY_PLANES[0]) | (1 << _XY_PLANES[1]))
        st_mask = mask & ~xy_mask
        out = {}
        lonlat = None
        for cache, sub, tag in ((self._stable_cache, st_mask, 'map_planes_dev'),
                                (self._cache, xy_mask, 'xy_map_dev')):
            if not sub:
                continue
            if tag == 'xy_map_dev' and not self._test_if_img_size_valid():
                raise ValueError('nx and ny must be positive to create a backplane image')
            key = (tag, mkey, alt)
            entry = cache.get(key)
            if entry is None or (entry[0] & sub) != sub:
                if lonlat is None:
                    lons, lats = self._get_lonlat_planes(**map_kwargs)
                    lonlat = (L.to_device(lons), L.to_device(lats))
                want = sub | (entry[0] if entry else 0)
                if tag == 'map_planes_dev':
                    want = L.ALL_PLANES & ~((1 << _XY_PLANES[0]) | (1 << _XY_PLANES[1]))
                else:
                    want = (1 << _XY_PLANES[0]) | (1 << _XY_PLANES[1])
                planes = L.backplanes_map_host(self._frame_host(alt), lonlat[0], lonlat[1], want)
                entry = (want, planes)
                cache[key] = entry
            out[tag] = entry
        return out

    def _get_map_plane(self, pid: int, **map_kwargs) -> np.ndarray:
        alt = self._check_alt(map_kwargs.get('alt', 0.0))
        mkey = self._map_key(map_kwargs)
        is_xy = pid in _XY_PLANES
        cache = self._cache if is_xy else self._stable_cache
        key = ('map_host', pid, mkey, alt)
        if key not in cache:
            tag = 'xy_map_dev' if is_xy else 'map_planes_dev'
            have, planes = self.get_backplanes_map_device(1 << pid, **map_kwargs)[tag]
            slot = L.popcount(have & ((1 << pid) - 1))
            cache[key] = _readonly(L.to_host(planes[slot]))
        return cache[key]

    def get_backplane_map(self, name: str, **map_kwargs) -> np.ndarray:
        """Copy of a backplane map (body_xy.py:2632-2663)."""
        bp = self.get_backplane_or_keyerror(name)
        if self._is_builtin_backplane(bp.name, mapped=True):
            pid = L.PLANE_ID[bp.name]
            tag = 'xy_map_dev' if pid in _XY_PLANES else 'map_planes_dev'
            have, planes = self.get_backplanes_map_device(1 << pid, **map_kwargs)[tag]
            return L.to_host(planes[L.popcount(have & ((1 << pid) - 1))])
        return np.array(bp.get_map(**map_kwargs), copy=True)

    # ---- image -> map resampling (body_xy.py:1414-1631) ---------------------------------
    def map_img(self, img, *, interpolation='linear', spline_smoothing: float = 0,
                propagate_nan: bool = True, warn_nan: bool = False,
                smooth_oversample_by: int = 5, smooth_max_oversampled_img_size: int = 10_000,
                **map_kwargs) -> np.ndarray:
        """Project an image (ny, nx) or cube (n, ny, nx) onto a lon/lat map."""
        out = self.map_img_device(img, interpolation=interpolation,
                                  spline_smoothing=spline_smoothing,
                                  propagate_nan=propagate_nan, warn_nan=warn_nan,
                                  smooth_oversample_by=smooth_oversample_by,
                                  smooth_max_oversampled_img_size=smooth_max_oversampled_img_size,
                                  **map_kwargs)
        res = L.to_host(out)
        return res[0] if np.ndim(img) == 2 else res

    @progress_decorator
    def map_img_device(self, img, *, interpolation='linear', spline_smoothing: float = 0,
                       propagate_nan: bool = True, warn_nan: bool = False, out=None,
                       smooth_oversample_by: int = 5, smooth_max_oversampled_img_size: int = 10_000,
                       **map_kwargs):
        """Same as :func:`map_img` but takes/returns device tensors shaped (n, ...)."""
        src = self._map_source(img, interpolation=interpolation, spline_smoothing=spline_smoothing,
                               propagate_nan=propagate_nan, warn_nan=warn_nan,
                               smooth_oversample_by=smooth_oversample_by,
                               smooth_max_oversampled_img_size=smooth_max_oversampled_img_size, **map_kwargs)
        return src.gather(0, src.n_planes, out=out)

    def _map_source(self, img, *, interpolation='linear', spline_smoothing: float = 0,
                    propagate_nan: bool = True, warn_nan: bool = False, smooth_oversample_by: int = 5,
                    smooth_max_oversampled_img_size: int = 10_000, **map_kwargs) -> '_MapSource':
        """Everything map_img needs ONCE per cube (body_xy.py:1571-1631): the cube on the device, the x / y
        maps of the requested projection and, for the spline modes, the repaired / prefiltered coefficient
        planes.  The result maps any range of planes on demand (one gather launch per call), which is how
        Observation walks a cube whose mapped output is larger than device or host memory."""
        smoothing = _smoothing_degrees(interpolation, spline_smoothing)
        torch = L._torch()
        mode = INTERP_REGRID if smoothing else _interpolation_mode(interpolation, spline_smoothing)
        if isinstance(img, torch.Tensor):
            cube = img if img.dim() == 3 else img[None]
            cube = cube.to(device='cuda', dtype=torch.float64).contiguous()
        else:
            arr = np.asarray(img)
            if arr.ndim not in (2, 3):
                raise ValueError(f'img must be 2D or 3D, got shape {arr.shape!r}')
            cube = L.to_device(arr if arr.ndim == 3 else arr[None])
        if tuple(cube.shape[1:]) != (self._ny, self._nx):
            raise ValueError(
                f'The input `img` shape {tuple(cube.shape[-2:])!r} is inconsistent with '
                f"the body's image size (ny={self._ny}, nx={self._nx})")
        have, xy = self.get_backplanes_map_device(
            (1 << _XY_PLANES[0]) | (1 << _XY_PLANES[1]), **map_kwargs)['xy_map_dev']
        spline = None
        if mode not in (L.INTERP_NEAREST, INTERP_SMOOTH):
            if warn_nan and bool(torch.isfinite(cube).logical_not().any()):
                print('Warning, image contains NaN values which will be corrected')
            if mode == INTERP_REGRID:
                spline = _fit_smoothing_splines(cube, *smoothing, spline_smoothing)
            else:
                spline = L.spline_prepare(cube, mode)
        return _MapSource(mode, cube, spline, xy[0], xy[1], propagate_nan, smooth_oversample_by,
                          smooth_max_oversampled_img_size)


class _MapSource:
    """A cube prepared for mapping onto one x / y map; ``gather(begin, count)`` maps planes
    [begin, begin + count) (``begin`` a multiple of 4 for the interpolating spline modes)."""

    def __init__(self, mode, cube, spline, xmap, ymap, propagate_nan, smooth_oversample_by, smooth_max_size):
        self.mode, self.cube, self.spline, self.xmap, self.ymap = mode, cube, spline, xmap, ymap
        self.propagate_nan = propagate_nan
        self.smooth_oversample_by, self.smooth_max_size = smooth_oversample_by, smooth_max_size
        self.n_planes = int(cube.shape[0])
        self.map_shape = tuple(xmap.shape)

    def gather(self, begin: int, count: int, out=None):
        if self.mode == L.INTERP_NEAREST:
            return L.gather(self.cube, self.xmap, self.ymap, self.mode, plane_begin=begin, plane_count=count, out=out)
        if self.mode == INTERP_SMOOTH:   # body_xy.py:1616-1629: planes are independent
            return L.map_smooth(self.cube[begin:begin + count], self.xmap, self.ymap, propagate_nan=self.propagate_nan,
                                oversample_by=self.smooth_oversample_by,
                                max_oversampled_img_size=self.smooth_max_size, out=out)
        if self.mode == INTERP_REGRID:
            return L.gather_regrid(self.spline, self.xmap, self.ymap, plane_begin=begin, plane_count=count,
                                   propagate_nan=self.propagate_nan, out=out)
        return L.gather(self.spline, self.xmap, self.ymap, self.mode, plane_begin=begin, plane_count=count,
                        propagate_nan=self.propagate_nan, out=out)


INTERP_SMOOTH = -1   # host-side marker: PCHIP oversampling + linear (its own entry points)
INTERP_REGRID = -2   # host-side marker: smoothing splines, spline_smoothing > 0 (pm_regrid_fit / pm_gather_regrid)

# scipy.interpolate._fitpack2._surfit_messages: RectBivariateSpline's ValueError text for each FITPACK ier
_SURFIT_MESSAGES = {1: """
The required storage space exceeds the available storage space: nxest
or nyest too small, or s too small.
The weighted least-squares spline corresponds to the current set of
knots.""",
                    2: """
A theoretically impossible result was found during the iteration
process for finding a smoothing spline with fp = s: s too small or
badly chosen eps.
Weighted sum of squared residuals does not satisfy abs(fp-s)/s < tol.""",
                    3: """
the maximal number of iterations maxit (set to 20 by the program)
allowed for finding a smoothing spline with fp=s has been reached:
s too small.
Weighted sum of squared residuals does not satisfy abs(fp-s)/s < tol.
Try increasing maxit by passing it as a keyword argument."""}


def _smoothing_degrees(interpolation, spline_smoothing):
    """(k_rows, k_cols) when map_img must fit smoothing splines (spline_smoothing != 0 with a spline degree),
    else None (every other call goes through _interpolation_mode unchanged)."""
    if spline_smoothing == 0:
        return None
    spline_k = {'linear': 1, 'quadratic': 2, 'cubic': 3}
    if isinstance(interpolation, str):
        if interpolation not in spline_k:
            return None
        k = spline_k[interpolation]
        degrees = (k, k)
    elif isinstance(interpolation, (int, np.integer)) and not isinstance(interpolation, bool):
        degrees = (int(interpolation), int(interpolation))
    elif isinstance(interpolation, tuple) and len(interpolation) == 2:
        degrees = tuple(int(k) for k in interpolation)
    else:
        return None
    if not all(1 <= k <= 3 for k in degrees):
        raise NotImplementedError(f'spline degrees {interpolation!r} with spline_smoothing != 0 are not '
                                  'accelerated (1..3 are)')
    if not spline_smoothing >= 0.0:   # RectBivariateSpline's own check
        raise ValueError('s should be s >= 0.0')
    return degrees


def _fit_smoothing_splines(cube, k_rows: int, k_cols: int, s: float):
    """RectBivariateSpline(arange(ny), arange(nx), plane, kx=k_rows, ky=k_cols, s=s) per plane on the device
    (body_xy.py:1651-1702); raises its ValueError for the first plane, in plane order, whose fit fails."""
    _, ny, nx = cube.shape
    if ny <= k_rows:
        raise ValueError('mx must be > kx')
    if nx <= k_cols:
        raise ValueError('my must be > ky')
    fit = L.regrid_fit(cube, k_rows, k_cols, float(s))
    bad = np.flatnonzero(~np.isin(fit.ier, (0, -1, -2)))
    if bad.size:
        ier = int(fit.ier[bad[0]])
        raise ValueError(_SURFIT_MESSAGES.get(ier, f'ier={ier}'))
    return fit


def _interpolation_mode(interpolation, spline_smoothing) -> int:
    spline_k = {'linear': 1, 'quadratic': 2, 'cubic': 3}
    if interpolation in spline_k:
        interpolation = spline_k[interpolation]
    if interpolation == 'nearest':
        return L.INTERP_NEAREST
    if isinstance(interpolation, tuple):
        # (kx, ky) as handed to RectBivariateSpline(np.arange(ny), np.arange(nx), img, kx=, ky=)
        # (body_xy.py:1673-1680): the FIRST degree runs along image rows (y)
        if len(interpolation) != 2:
            raise ValueError(f'Unknown interpolation method {interpolation!r}')
        if spline_smoothing != 0:
            raise NotImplementedError('spline_smoothing != 0 (FITPACK smoothing) is not '
                                      'accelerated; only interpolating splines are')
        k_rows, k_cols = (int(k) for k in interpolation)
        if not (1 <= k_rows <= 3 and 1 <= k_cols <= 3):
            raise NotImplementedError(f'spline degrees {interpolation!r} are not accelerated (1..3 are)')
        if k_rows == k_cols:
            return k_rows
        return L.INTERP_MIXED | (k_rows << 4) | k_cols
    if isinstance(interpolation, (int, np.integer)) and not isinstance(interpolation, bool):
        if spline_smoothing != 0:
            raise NotImplementedError('spline_smoothing != 0 (FITPACK smoothing) is not '
                                      'accelerated; only interpolating splines are')
        if interpolation == 1:
            return L.INTERP_LINEAR
        if interpolation == 2:
            return L.INTERP_QUADRATIC
        if interpolation == 3:
            return L.INTERP_CUBIC
        raise NotImplementedError(
            f'spline degree {interpolation} is not accelerated (SURVEY.md 8(f)); '
            "accelerated: 'nearest', 'linear' (1), 'quadratic' (2), 'cubic' (3)")
    if interpolation == 'smooth':
        return INTERP_SMOOTH
    raise ValueError(f'Unknown interpolation method {interpolation!r}')


class _AltitudeScope:
    """_AdjustedSurfaceAltitude (body.py:172-229) without the kernel-pool mutation:
    the adjusted radii travel inside the PMFrame."""

    def __init__(self, body: BodyXY, alt: float = 0.0) -> None:
        self.body = body
        self.alt = float(alt)
        self.active = self.alt != 0.0 and self.alt != body._alt_adjustment
        if self.active and body._alt_adjustment != 0.0:
            raise ValueError('Cannot nest altitude adjustments with alt != 0')

    def __enter__(self) -> None:
        if self.active:
            self.body._alt_adjustment = self.alt

    def __exit__(self, *exc) -> None:
        if self.active:
            self.body._alt_adjustment = 0.0
