"""Shared comparison helpers for the parity tests."""
import numpy as np

from planetmapper_b200 import frame as F

PLANE_NAMES = [
    'LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'RA', 'DEC', 'PIXEL-X',
    'PIXEL-Y', 'KM-X', 'KM-Y', 'ANGULAR-X', 'ANGULAR-Y', 'PHASE', 'INCIDENCE',
    'EMISSION', 'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER',
    'LIMB-DISTANCE', 'LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC', 'RING-RADIUS',
    'RING-LON-GRAPHIC', 'RING-DISTANCE',
]
PID = {n: i for i, n in enumerate(PLANE_NAMES)}
ANGLE_PLANES = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE',
                'EMISSION', 'AZIMUTH']


def angle_diff(a, b):
    """|a - b| in degrees, treating 0 / 360 as the same longitude."""
    d = np.abs(a - b)
    return np.minimum(d, np.abs(360.0 - d))


def max_diff(a, b, wrap=False):
    ok = np.isfinite(a) & np.isfinite(b)
    if not ok.any():
        return 0.0
    d = angle_diff(a[ok], b[ok]) if wrap else np.abs(a[ok] - b[ok])
    return float(d.max())


def masks_equal(a, b, exclude=None):
    """NaN masks identical outside `exclude`; returns (ok, n_mismatch, n_excluded)."""
    mism = np.isnan(a) != np.isnan(b)
    n_ex = 0
    if exclude is not None:
        n_ex = int((mism & exclude).sum())
        mism = mism & ~exclude
    return (not mism.any()), int(mism.sum()), n_ex


def lst_boundary(lon_deg, frame_lon_sign, sun_lon, prograde=True, tol_s=1e-6):
    """True where the local-solar-time second count is within tol_s of an integer
    boundary (LOCAL-SOLAR-TIME is quantised to whole seconds: body.py:2397-2398)."""
    ang = frame_lon_sign * np.deg2rad(lon_deg) - sun_lon
    if not prograde:
        ang = -ang
    ang = np.mod(ang, 2 * np.pi)
    sec = ang * (86400.0 / (2 * np.pi)) + 43200.0
    frac = sec - np.floor(sec)
    return (frac < tol_s) | (frac > 1 - tol_s)


# ---------------------------------------------------------------------------------
# Conditioning-aware tolerances for the image-direction surface planes.
#
# north_star's bars are 1e-9 deg (angles) and 1e-12 relative (distances, velocities).
# The reference itself cannot deliver that near the limb: CSPICE forms the observer
# position in the body frame with magnitude |P0| ~ 8e8 km, i.e. with a rounding
# granularity ulp(|P0|) ~ 1.2e-7 km, and a perpendicular error d of the ray moves the
# intercept by d / cos(emission) along the surface.  Two correct FP64 evaluations
# (different operation order, FMA contraction) therefore differ by about
# 2 ulp(|P0|) / (r cos e) radians.  The tolerances below are the stated bars, widened
# ONLY by that amplification factor kappa = 1 / cos(emission) where it exceeds them.
# ---------------------------------------------------------------------------------
def surface_tolerances(ref_planes, p0_norm, r_min, omega_norm, epoch_quantum_km=0.0):
    emi = ref_planes[PID['EMISSION']]
    latc = ref_planes[PID['LAT-CENTRIC']]
    with np.errstate(invalid='ignore', divide='ignore'):
        kappa = 1.0 / np.maximum(np.cos(np.deg2rad(emi)), 1e-12)
        # km, positional rounding noise (+ optionally one epoch quantum of relative motion, see
        # check_img_planes)
        delta = 2.0 * np.spacing(p0_norm) + epoch_quantum_km
        ang = np.rad2deg(delta * kappa / r_min)           # deg, induced angle noise
        base = np.maximum(1e-9, 4.0 * ang)
        coslat = np.maximum(np.cos(np.deg2rad(latc)), 1e-12)
    tol = {
        'LAT-GRAPHIC': base, 'LAT-CENTRIC': base, 'INCIDENCE': base, 'EMISSION': base,
        'LON-GRAPHIC': base / coslat, 'LON-CENTRIC': base / coslat,
        'PHASE': np.full_like(base, 1e-9),
        # a lateral shift d of the ray moves the intercept by d tan(e) along the line of sight
        'DISTANCE': 1e-12 * p0_norm + 2.0 * delta * kappa,
        'RADIAL-VELOCITY': 1e-12 * np.abs(ref_planes[PID['RADIAL-VELOCITY']]) + 4.0 * omega_norm * delta * kappa + 1e-13,
    }
    tol['DOPPLER'] = tol['RADIAL-VELOCITY'] / 299792.458 + 4e-16
    # AZIMUTH is a float64 formula of (phase, incidence, emission) that is itself
    # ill-conditioned near the sub-observer / sub-solar points: propagate numerically
    g, i, e = (np.deg2rad(ref_planes[PID[n]]) for n in ('PHASE', 'INCIDENCE', 'EMISSION'))
    t = np.deg2rad(base)

    def az(g, i, e):
        with np.errstate(invalid='ignore', divide='ignore'):
            a = np.cos(g) - np.cos(e) * np.cos(i)
            b = np.sqrt(1.0 - np.cos(e) ** 2) * np.sqrt(1.0 - np.cos(i) ** 2)
            return np.rad2deg(np.pi - np.arccos(np.clip(a / b, -1, 1)))

    az0 = az(g, i, e)
    dev = np.zeros_like(base)
    for sg in (-1, 1):
        for si in (-1, 1):
            for se in (-1, 1):
                with np.errstate(invalid='ignore'):
                    dev = np.fmax(dev, np.abs(az(g + sg * np.deg2rad(1e-9), i + si * t, e + se * t) - az0))
    tol['AZIMUTH'] = 2.0 * dev + 1e-9
    return tol, kappa


# ---------------------------------------------------------------------------------
# Shared cases and plane-by-plane comparisons (used by the GPU parity tests and by the
# host instantiation of the device code, tests/test_host_check.py)
# ---------------------------------------------------------------------------------
WRAP = {'LON-GRAPHIC', 'LON-CENTRIC', 'LIMB-LON-GRAPHIC', 'RING-LON-GRAPHIC'}
SURFACE = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE', 'EMISSION',
           'AZIMUTH', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER']


def img_case(bc, nx, ny, x0, y0, r0, rot_deg, alt=0.0):
    return F.pack_frame(bc, nx=nx, ny=ny, x0=x0, y0=y0, r0=r0, rotation_radians=np.deg2rad(rot_deg), alt=alt)


IMG_CASES = {
    'golden-7x10': (7, 10, 2.5, 3.1, 3.9, 123.456, 0.0),
    'golden-7x10-alt': (7, 10, 2.5, 3.1, 3.9, 123.456, 34567.8912),
    'C1-100x100': (100, 100, 49.5, 49.5, 44.55, 0.0, 0.0),
    'rot-200x160': (200, 160, 99.5, 79.5, 70.0, 30.0, 0.0),
    'offset-disc-partly-outside': (64, 48, 50.0, 10.0, 40.0, 200.0, 0.0),
    'ragged-1x37': (1, 37, 0.0, 18.0, 12.0, 0.0, 0.0),
}


def epoch_quantum_km(fr):
    """CSPICE forms every point epoch as et - lt in FP64: granularity ulp(et) ~ 3e-8 s.  The
    target is evaluated at that epoch while the observer stays at et, so one quantum moves
    the target by |V_target| ulp(et) ~ 1e-6 km (barycentric speed, ~13 km/s for Jupiter,
    ~30 km/s for the inner planets and the Moon).  Both the oracle and the kernels carry that
    noise relative to an extended-precision evaluation of the same algorithm
    (tests/test_host_check.py::test_device_code_vs_extended_precision measures it), and two
    FP64 evaluations land on different quanta in a few pixels per thousand."""
    v = float(np.linalg.norm(F.frame_field(fr, 'VT')))
    return v * float(np.spacing(F.frame_field(fr, 'et')[0]))


OTHER_BODIES = [
    # target, observer, nx, ny, x0, y0, r0, rotation: branches the Jupiter fixture never takes
    ('Venus', 'EARTH', 80, 64, 40.0, 30.0, 25.0, 15.0),    # retrograde spin (et2lst sign), sphere
    ('Moon', 'EARTH', 72, 72, 35.5, 35.5, 30.0, -20.0),    # near field (0.5 deg disc), sphere, east-positive
    ('Earth', 'MOON', 64, 80, 30.0, 41.0, 26.0, 200.0),    # 1.9 deg disc, oblate, east-positive
    ('Mars', 'EARTH', 90, 60, 44.5, 29.5, 24.0, 5.0),      # west-positive prograde, small flattening
    ('Mercury', 'EARTH', 48, 48, 23.5, 23.5, 18.0, 90.0),
]



# ---------------------------------------------------------------------------------
# Triaxial bodies (BASELINE config C5 names Europa: 1562.6 / 1560.3 / 1559.5 km).  The bundled
# kernels have no SPK segment for 502, so its position comes from an analytic orbit about the
# Jupiter barycentre (planetmapper_b200/minispice/kepler.py, SURVEY 8(d) C5 option ii); radii and
# the IAU orientation model are the PCK's.  'triaxial-x' keeps Europa's state and orientation but
# exaggerates the shape so that every triaxial term (sincpt on (a, b, c), surfnm weights, recpgr
# against (a, a, c) of a point OFF that spheroid, pgrrec points off the ellipsoid) is far above
# rounding level.
# ---------------------------------------------------------------------------------
class _RadiiOverride:
    def __init__(self, base, body, radii):
        self.base, self.body, self.radii = base, int(body), np.asarray(radii, dtype=float)

    def __getattr__(self, item):
        return getattr(self.base, item)

    def bodvar(self, body, item):
        if int(body) == self.body and item == 'RADII':
            return self.radii.copy()
        return self.base.bodvar(body, item)


def triaxial_constants(kind='europa', utc='2004-12-31T00:00:00', observer='EARTH'):
    import planetmapper_b200 as pm
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    provider = KeplerOrbitProvider(pm.get_default_provider())
    if kind == 'triaxial-x':
        provider = _RadiiOverride(provider, 502, [1562.6, 1420.3, 1260.5])
    bc = F.build_body_constants(provider, 'Europa', utc, observer)
    assert len(set(bc.radii)) == 3
    return bc


def close_observer_constants(utc='2005-01-01T03:00:00'):
    """Jupiter from Amalthea (synthetic two-body orbit, minispice/kepler.py): observer 2.5 radii out."""
    import planetmapper_b200 as pm
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    return F.build_body_constants(KeplerOrbitProvider(pm.get_default_provider()), 'Jupiter', utc, 'AMALTHEA')


def random_geometry(seed):
    """A random frame for the referee tests: target among six bodies (oblate, spherical, triaxial, retrograde,
    fast and slow rotators), observer anywhere between 1.3 and 1e5 body radii in a random direction with a
    random velocity of up to ~50 km/s relative to the target, random disc position / size / rotation.
    Returns (frame, nx, ny, label)."""
    bc, disc, alt, label = random_geometry_parts(seed)
    return img_case(bc, *disc, alt), disc[0], disc[1], label


def random_geometry_parts(seed):
    """random_geometry(seed) before packing: (constants, (nx, ny, x0, y0, r0, rotation in degrees), alt, label)."""
    import planetmapper_b200 as pm
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    prov = KeplerOrbitProvider(pm.get_default_provider())
    rng = np.random.default_rng(seed)
    target = ['Jupiter', 'Saturn', 'Moon', 'Europa', 'Mars', 'Venus'][rng.integers(6)]
    utc = '2004-12-%02dT%02d:00:00' % (rng.integers(27, 31), rng.integers(0, 24))
    et = prov.utc2et(utc)
    tid = prov.bods2c(target)
    tstate = prov.ssb_state(tid, et)
    rmax = float(max(prov.bodvar(tid, 'RADII')))
    dist = rmax * 10 ** rng.uniform(np.log10(1.3), 5)
    n = rng.normal(size=3)
    n /= np.linalg.norm(n)
    v = rng.normal(size=3) * rng.uniform(0, 30)
    obs = np.concatenate([tstate[:3] + dist * n, tstate[3:] + v])
    bc = F.build_body_constants(prov, target, utc, 'EARTH', observer_state=obs)
    nx, ny = int(rng.integers(40, 120)), int(rng.integers(40, 120))
    r0 = rng.uniform(0.2, 0.9) * min(nx, ny)
    x0, y0 = rng.uniform(0.2, 0.8) * nx, rng.uniform(0.2, 0.8) * ny
    rot = rng.uniform(0, 360)
    # every fourth geometry on an altitude-adjusted surface (get_backplane_img(..., alt=...), body_xy.py:2586)
    alt = float(rng.uniform(-0.01, 0.05) * rmax) if seed % 4 == 3 else 0.0
    return (bc, (nx, ny, x0, y0, r0, rot), alt,
            f'seed {seed}: {target} D/r={dist / rmax:.3g} {nx}x{ny} r0={r0:.1f} rot={rot:.0f} alt={alt:.0f}')


def referee_ratios(got, ref, exact, margin, xy_floor=None):
    """For every continuous plane: how far `got` (kernel code) and `ref` (FP64 oracle) each sit from `exact`
    (the oracle in 80-bit arithmetic), as (max ratio, rms ratio) of got-vs-exact over ref-vs-exact.  The
    denominators are floored at north_star's bare bars (1e-9 deg, 1e-12 relative; a tenth of them for the
    rms): below those both are inside the bar and the ratio says nothing.  xy_floor (pixels) switches the
    PIXEL-X / PIXEL-Y planes on - the x / y maps of the map direction - with that floor."""
    grazing = np.where(np.isnan(margin), False, np.abs(margin) < 1e-9)
    out = {}
    for name in PLANE_NAMES:
        if name == 'LOCAL-SOLAR-TIME' or (name in ('PIXEL-X', 'PIXEL-Y') and xy_floor is None):
            continue   # integer seconds; pixel indices in the image direction
        k = PID[name]
        both = np.isfinite(got[k]) & np.isfinite(ref[k]) & np.isfinite(exact[k]) & ~grazing
        if not both.any():
            continue
        diff = angle_diff if name in WRAP else (lambda a, b: np.abs(a - b))
        de, oe = diff(got[k], exact[k])[both], diff(ref[k], exact[k])[both]
        floor = 1e-9 if name in BARE_ANGLE_PLANES else 1e-12 * float(np.abs(exact[k][both]).max())
        if name in ('PIXEL-X', 'PIXEL-Y'):
            floor = xy_floor   # x_map / y_map of the map direction, pixels
        out[name] = (float(de.max() / max(oe.max(), floor)),
                     float(np.sqrt(np.mean(de ** 2)) / max(np.sqrt(np.mean(oe ** 2)), 0.1 * floor)),
                     float(de.max()), float(oe.max()))
    return out


def assert_referee(got, ref, exact, margin, label, xy_floor=None):
    """The kernel code is as close to the extended-precision result as the FP64 oracle is: rms within 3x,
    worst pixel within 10x (a maximum over a few thousand pixels of two independent rounding-noise fields;
    420 random geometries give <= 7.8x and <= 2.9x rms outside the two limb-angle planes, see below), NaN masks
    identical outside grazing pixels."""
    grazing = np.where(np.isnan(margin), False, np.abs(margin) < 1e-9)
    for name in PLANE_NAMES:
        ok, n_bad, _ = masks_equal(got[PID[name]], ref[PID[name]], exclude=grazing)
        assert ok, f'{label} {name}: {n_bad} NaN-mask mismatches outside grazing pixels'
    rr = referee_ratios(got, ref, exact, margin, xy_floor)
    for name, (r_max, r_rms, d_max, o_max) in rr.items():
        # LIMB-LON / LIMB-LAT: the limb point is the radial projection of the ray's closest approach to the body
        # centre, a difference of two |P0|-sized vectors - a ray through the centre has no defined limb point at
        # all, and the worst pixel of a frame is whichever ray passes nearest to it (324 further geometries: up to
        # 13x in the maximum, 4.9x rms, with both errors below 5e-8 deg)
        lim_max, lim_rms = (30.0, 6.0) if name in ('LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC') else (10.0, 3.0)
        assert r_rms <= lim_rms and r_max <= lim_max, (
            f'{label} {name}: kernel-vs-exact / oracle-vs-exact = {r_max:.2f} (max), {r_rms:.2f} (rms); '
            f'max errors {d_max:.3e} / {o_max:.3e}')
    return rr


TRIAXIAL_CASES = [
    # kind, nx, ny, x0, y0, r0, rotation
    ('europa', 96, 80, 47.5, 40.0, 33.0, 25.0),
    ('triaxial-x', 96, 80, 47.5, 40.0, 33.0, 25.0),
    ('triaxial-x', 64, 64, 20.0, 40.0, 45.0, 250.0),    # disc partly outside the frame
]


# north_star's bars as written, with no conditioning term: angles 1e-9 deg, distances and
# velocities 1e-12 relative.  raw_plane_stats() reports every compared pixel against them.
BARE_ANGLE_PLANES = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE', 'EMISSION',
                     'AZIMUTH', 'RA', 'DEC', 'LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC', 'RING-LON-GRAPHIC']
BARE_REL_PLANES = ['DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER', 'LIMB-DISTANCE', 'RING-RADIUS', 'RING-DISTANCE']
EMISSION_BINS = [0.0, 35.0, 60.0, 80.0, 89.0, 90.0]


def raw_plane_stats(got, ref, margin, planes=None):
    """Un-widened statistics of `got` against `ref` (26-plane stacks; absent planes all-NaN): per plane
    the number of pixels compared, the maximum difference, how many pixels exceed the BARE bar
    (1e-9 deg / 1e-12 relative) and where they sit in emission angle.  Nothing is asserted here."""
    grazing = np.where(np.isnan(margin), False, np.abs(margin) < 1e-9)
    emi = ref[PID['EMISSION']]
    out = {'n_px': int(got[0].size), 'n_grazing_excluded': int(grazing.sum())}
    for name in (planes or BARE_ANGLE_PLANES + BARE_REL_PLANES + ['LOCAL-SOLAR-TIME']):
        a, b = got[PID[name]], ref[PID[name]]
        both = np.isfinite(a) & np.isfinite(b) & ~grazing
        mism = (np.isnan(a) != np.isnan(b))
        if not both.any() and not mism.any():
            continue
        d = angle_diff(a, b) if name in WRAP else np.abs(a - b)
        if name in BARE_REL_PLANES:
            with np.errstate(invalid='ignore', divide='ignore'):
                d = d / np.abs(b)
            bar, unit = 1e-12, 'relative'
        elif name == 'LOCAL-SOLAR-TIME':
            bar, unit = 0.0, 'hours (integer seconds: exact or one second off at a boundary)'
        else:
            bar, unit = 1e-9, 'deg'
        dd = np.where(both, d, 0.0)
        over = both & (dd > bar)
        entry = {'unit': unit, 'bare_bar': bar, 'n_compared': int(both.sum()), 'max_diff': float(dd.max()),
                 'n_over_bare_bar': int(over.sum()), 'frac_over_bare_bar': float(over.sum() / max(1, both.sum())),
                 'mask_mismatch_outside_grazing': int((mism & ~grazing).sum()),
                 'mask_mismatch_in_grazing': int((mism & grazing).sum())}
        if over.any() and np.isfinite(emi[over]).any():
            hist, _ = np.histogram(emi[over], bins=EMISSION_BINS)
            entry['over_by_emission_bin'] = {f'{lo:g}-{hi:g}': int(n) for lo, hi, n in
                                             zip(EMISSION_BINS[:-1], EMISSION_BINS[1:], hist)}
            entry['min_emission_of_over_deg'] = float(np.nanmin(emi[over]))
        out[name] = entry
    return out


def write_parity_report(key, stats):
    """Merges `stats` into gpurun_out/parity_report.json (scratch; the committed copy is
    profiles/parity_c2_c3.json)."""
    import json
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = os.path.join(root, 'gpurun_out', 'parity_report.json')
    os.makedirs(os.path.dirname(path), exist_ok=True)
    data = {}
    if os.path.exists(path):
        try:
            with open(path) as f:
                data = json.load(f)
        except ValueError:
            data = {}
    data[key] = stats
    with open(path, 'w') as f:
        json.dump(data, f, indent=1)


def check_img_planes(got, ref, margin, fr, label, allow_epoch_quantum=False):
    """Shared comparison of 26 image-direction planes (GPU `got` vs oracle `ref`).
    allow_epoch_quantum widens the positional noise term by one epoch quantum (used for
    the bodies outside BASELINE.json's configs, whose |P0| / r conditioning is worse; the
    named Jupiter / Saturn configs are held to the bare bar)."""
    grazing = np.abs(margin) < 1e-9
    grazing = np.where(np.isnan(margin), False, grazing)
    p0 = float(np.linalg.norm(F.frame_field(fr, 'P0')))
    r_min = float(np.min(F.frame_field(fr, 'radii')))
    w = float(np.linalg.norm(F.frame_field(fr, 'omega')))
    tol, kappa = surface_tolerances(ref, p0, r_min, w, epoch_quantum_km(fr) if allow_epoch_quantum else 0.0)
    report = {}
    n_grazing_mismatch = 0
    for name in PLANE_NAMES:
        a, b = got[PID[name]], ref[PID[name]]
        ok, n_bad, n_ex = masks_equal(a, b, exclude=grazing)
        n_grazing_mismatch = max(n_grazing_mismatch, n_ex)
        assert ok, f'{label} {name}: {n_bad} NaN-mask mismatches outside grazing pixels'
        both = np.isfinite(a) & np.isfinite(b) & ~grazing
        if not both.any():
            continue
        d = angle_diff(a, b) if name in WRAP else np.abs(a - b)
        if name in tol:
            ratio = np.max(d[both] / tol[name][both])
            report[name] = ratio
            assert ratio <= 1.0, f'{label} {name}: diff/tol = {ratio:.3f} (max diff {np.max(d[both]):.3e})'
        elif name == 'LOCAL-SOLAR-TIME':
            lon_tol = tol['LON-GRAPHIC']
            boundary = lst_boundary(ref[PID['LON-GRAPHIC']], F.frame_field(fr, 'lon_sign')[0],
                                    F.frame_field(fr, 'sun_lon_lst')[0], tol_s=1e-6) | \
                (240.0 * lon_tol > 1e-6) & lst_boundary(ref[PID['LON-GRAPHIC']], F.frame_field(fr, 'lon_sign')[0],
                                                        F.frame_field(fr, 'sun_lon_lst')[0], tol_s=1e-4)
            sel = both & ~boundary
            assert np.array_equal(a[sel], b[sel]), f'{label} LST differs away from second boundaries'
            # at a boundary the value may flip by exactly one second
            flip = both & boundary & (a != b)
            assert np.all(np.abs(a[flip] - b[flip]) < 1.5 / 3600), label
        elif name in ('RA', 'DEC'):
            assert np.max(d[both]) <= 1e-12, f'{label} {name}: {np.max(d[both]):.3e}'
        elif name in ('PIXEL-X', 'PIXEL-Y'):
            assert np.array_equal(a[both], b[both])
        elif name in ('KM-X', 'KM-Y'):
            # 1e-5 km at the named configs; 1e-12 relative for wide fields, and never below the RA / Dec
            # round trip in degrees the reference goes through (ulp(360 deg) of sky at the target's distance)
            t = max(1e-5, 1e-12 * float(np.max(np.abs(b[both]))), 4.0 * np.deg2rad(np.spacing(360.0)) * p0)
            assert np.max(d[both]) <= t, f'{label} {name}: {np.max(d[both]):.3e} km'
        elif name in ('ANGULAR-X', 'ANGULAR-Y'):
            t = max(1e-8, 1e-12 * float(np.max(np.abs(b[both]))))
            assert np.max(d[both]) <= t, f'{label} {name}: {np.max(d[both]):.3e} arcsec'
        elif name in ('RING-DISTANCE', 'RING-RADIUS'):
            assert np.max(d[both]) <= 1e-12 * p0 * 50, f'{label} {name}: {np.max(d[both]):.3e} km'
        elif name == 'RING-LON-GRAPHIC':
            # ray / ring-plane intercept: a perpendicular ray error is stretched by
            # 1 / sin(opening angle) = RING-DISTANCE / ring_c along the plane
            rr = np.abs(ref[PID['RING-RADIUS']])
            stretch = np.abs(ref[PID['RING-DISTANCE']]) / F.frame_field(fr, 'ring_c')[0]
            t = np.maximum(1e-9, np.rad2deg(8 * np.spacing(p0) * stretch / np.maximum(rr, 1.0)))
            assert np.all(d[both] <= t[both]), f'{label} {name}: {np.max(d[both]):.3e}'
        elif name.startswith('LIMB'):
            # the limb point is the radial projection of the ray's closest approach to
            # the centre: conditioning ~ r / (distance of closest approach)
            # (projected distance of the ray from the body centre = |(KM-X, KM-Y)|; a ray
            # through the centre has no defined limb longitude / latitude at all)
            near = np.hypot(ref[PID['KM-X']], ref[PID['KM-Y']])
            cond = np.maximum(1.0, r_min * 1.2 / np.maximum(near, 1e-3))
            if name == 'LIMB-DISTANCE':
                assert np.max(d[both]) <= 1e-12 * p0 * 50, f'{label} {name}: {np.max(d[both]):.3e} km'
            else:
                t = np.maximum(1e-9, np.rad2deg(16 * np.spacing(p0) / r_min) * cond)
                if name == 'LIMB-LON-GRAPHIC':
                    t = t / np.maximum(np.cos(np.deg2rad(ref[PID['LIMB-LAT-GRAPHIC']])), 1e-9)
                assert np.all(d[both] <= t[both]), f'{label} {name}: {np.max(d[both] / t[both]):.3f}'
    return report, int(grazing.sum()), n_grazing_mismatch


def check_map_planes(got, ref, margin, fr, nx, ny, case):
    """Shared comparison of 26 map-direction planes (`got` vs oracle `ref`)."""
    grazing = np.where(np.isnan(margin), False, np.abs(margin) < 1e-9)
    # also cells grazing the terminator (`lit` drives the LIMB / RING maps)
    graz_lit = np.where(np.isnan(ref[PID['INCIDENCE']]), False, np.abs(ref[PID['INCIDENCE']] - 90.0) < 1e-7)
    p0 = float(np.linalg.norm(F.frame_field(fr, 'P0')))
    for name in PLANE_NAMES:
        a, b = got[PID[name]], ref[PID[name]]
        ex = grazing | graz_lit if (name.startswith('LIMB') or name.startswith('RING')) else grazing
        if name in ('PIXEL-X', 'PIXEL-Y'):
            # cells within 1e-9 px of the image frame edge may flip (counted, not hidden)
            x, y = ref[PID['PIXEL-X']], ref[PID['PIXEL-Y']]
            gx, gy = got[PID['PIXEL-X']], got[PID['PIXEL-Y']]
            edge = np.zeros(x.shape, dtype=bool)
            for v, n in ((np.where(np.isnan(x), gx, x), nx), (np.where(np.isnan(y), gy, y), ny)):
                with np.errstate(invalid='ignore'):
                    edge |= (np.abs(v + 0.5) < 1e-9) | (np.abs(v - (n - 0.5)) < 1e-9)
            ex = ex | edge
        ok, n_bad, _ = masks_equal(a, b, exclude=ex)
        assert ok, f'{case} map {name}: {n_bad} mask mismatches'
        both = np.isfinite(a) & np.isfinite(b)
        if not both.any():
            continue
        d = angle_diff(a, b) if name in WRAP else np.abs(a - b)
        m = float(np.max(d[both]))
        if name in ('LON-GRAPHIC', 'LAT-GRAPHIC', 'LOCAL-SOLAR-TIME'):
            assert m == 0.0, (case, name, m)
        elif name in ('LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE', 'EMISSION', 'RA', 'DEC'):
            assert m <= 1e-9, (case, name, m)
        elif name == 'AZIMUTH':
            tol, _ = surface_tolerances(ref, p0, 6e4, 1.8e-4)
            assert np.all(d[both] <= np.maximum(tol['AZIMUTH'][both], 1e-9)), (case, name, m)
        elif name in ('DISTANCE', 'RING-DISTANCE', 'RING-RADIUS', 'LIMB-DISTANCE'):
            assert m <= 1e-12 * p0 * 50, (case, name, m)
        elif name in ('RADIAL-VELOCITY', 'DOPPLER'):
            # CSPICE forms the point epoch et - lt in FP64 (granularity ulp(et) ~ 3e-8 s);
            # two converged light times that differ in the last bit can land on either
            # side of it, which moves the rotational velocity by omega^2 r ulp(et)
            w = float(np.linalg.norm(F.frame_field(fr, 'omega')))
            r_max = float(np.max(F.frame_field(fr, 'radii')))
            et_quantum = w * w * r_max * float(np.spacing(F.frame_field(fr, 'et')[0]))
            rv_tol = 1e-12 * 40 + 2e-13 + et_quantum
            if name == 'DOPPLER':
                assert m <= rv_tol / 299792.458 + 4e-16, (case, name, m)
            else:
                assert m <= rv_tol, (case, name, m)
        elif name in ('PIXEL-X', 'PIXEL-Y'):
            assert m <= 1e-9 * max(nx, ny), (case, name, m)   # <= 1e-9 deg on the sky
        elif name in ('KM-X', 'KM-Y'):
            assert m <= 1e-5, (case, name, m)
        elif name in ('ANGULAR-X', 'ANGULAR-Y'):
            assert m <= 1e-8, (case, name, m)
