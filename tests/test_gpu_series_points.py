"""
GPU tests of the point transforms over the epochs of a time series (planetmapper_b200.series.transform):
every row of one batched launch against a fresh BodyXY per epoch, with that epoch's own disc parameters,
calling the matching public method - bit for bit, NaN masks included.
"""
import numpy as np
import pytest

from planetmapper_b200 import frame as F

pytestmark = pytest.mark.gpu

# BodyXY method -> (src, dst, keyword groups it accepts): alt, nvn = not_visible_nan, nfn = not_found_nan,
# pc = planetocentric, ang = origin_ra / origin_dec / coordinate_rotation
METHODS = {
    'xy2lonlat': ('xy', 'lonlat', {'alt', 'nfn', 'pc'}),
    'lonlat2xy': ('lonlat', 'xy', {'alt', 'nvn', 'pc'}),
    'xy2radec': ('xy', 'radec', set()),
    'radec2xy': ('radec', 'xy', set()),
    'xy2km': ('xy', 'km', set()),
    'km2xy': ('km', 'xy', set()),
    'xy2angular': ('xy', 'angular', {'ang'}),
    'angular2xy': ('angular', 'xy', {'ang'}),
    'lonlat2radec': ('lonlat', 'radec', {'alt', 'nvn', 'pc'}),
    'radec2lonlat': ('radec', 'lonlat', {'alt', 'nfn', 'pc'}),
    'radec2angular': ('radec', 'angular', {'ang'}),
    'angular2radec': ('angular', 'radec', {'ang'}),
    'angular2lonlat': ('angular', 'lonlat', {'alt', 'nfn', 'pc', 'ang'}),
    'lonlat2angular': ('lonlat', 'angular', {'alt', 'nvn', 'pc', 'ang'}),
    'km2radec': ('km', 'radec', set()),
    'radec2km': ('radec', 'km', set()),
    'km2lonlat': ('km', 'lonlat', {'alt', 'nfn', 'pc'}),
    'lonlat2km': ('lonlat', 'km', {'alt', 'nvn', 'pc'}),
    'km2angular': ('km', 'angular', {'ang'}),
    'angular2km': ('angular', 'km', {'ang'}),
    'graphic2centric_lonlat': ('lonlat', 'centric', {'alt'}),
    'centric2graphic_lonlat': ('lonlat', 'lonlat', {'alt'}),
}
NX, NY = 40, 30


class Series:
    """A series built with per-epoch disc parameters, and the BodyXY of every epoch."""

    def __init__(self, target, ets, provider, workers, kepler=False):
        import planetmapper_b200 as pm
        from planetmapper_b200 import series as S
        from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

        n = len(ets)
        k = np.arange(n)
        self.x0 = 19.5 + 1.7 * np.sin(0.9 * k)          # pointing drift
        self.y0 = 14.5 - 0.45 * k + 0.2 * np.cos(k)
        self.r0 = 11.0 + 0.13 * k                          # the disc grows as the target approaches
        rot_deg = 20.0 + 3.5 * k
        self.rot_deg = rot_deg
        self.rot_rad = np.array([float(np.deg2rad(float(r))) % (2 * np.pi) for r in rot_deg])   # BodyXY.set_rotation
        series_provider = None if workers > 1 else provider
        self.frames, self.k2a = S.build_series_frames(
            target, ets, 'EARTH', nx=NX, ny=NY, x0=self.x0, y0=self.y0, r0=self.r0, rotation_radians=self.rot_rad,
            workers=workers, provider=series_provider, kepler=kepler, with_km2angular=True)
        prov = KeplerOrbitProvider(provider) if kepler else provider
        self.bodies = []
        for f, et in enumerate(ets):
            body = pm.BodyXY(nx=NX, ny=NY, constants=F.build_body_constants(prov, target, None, 'EARTH', et=float(et)))
            body.set_disc_params(self.x0[f], self.y0[f], self.r0[f], rot_deg[f])
            assert np.array_equal(body._frame_host(), self.frames[f])   # the series frame IS the epoch's frame
            self.bodies.append(body)


@pytest.fixture(scope='module')
def jupiter():
    import planetmapper_b200 as pm
    from planetmapper_b200 import series as S

    prov = pm.get_default_provider()
    # 32 epochs, so that workers=2 really shards (a block under 16 epochs runs serially)
    ets = prov.utc2et('2005-01-01T00:00:00') + 5400.0 * np.arange(32)
    try:
        yield Series('Jupiter', ets, prov, workers=2)
    finally:
        S.shutdown_pool()


@pytest.fixture(scope='module')
def europa():
    import planetmapper_b200 as pm

    prov = pm.get_default_provider()
    ets = prov.utc2et('2004-12-30T00:00:00') + 1800.0 * np.arange(8)
    return Series('Europa', ets, prov, workers=1, kepler=True)


def _inputs(ser, src):
    """Points of system ``src`` on the disc, on the limb, off the disc and in the sky, plus NaN / inf entries:
    (shared (n,), per-frame (n_frames, n))."""
    xs, ys = np.meshgrid(np.linspace(-3.0, NX + 2.0, 17), np.linspace(-2.5, NY + 1.5, 13))
    xy = (xs.ravel(), ys.ravel())
    b0 = ser.bodies[0]
    if src == 'xy':
        a, b = xy
    elif src == 'lonlat':
        lo, la = np.meshgrid(np.arange(0.0, 360.0, 23.0), np.arange(-88.0, 90.0, 16.0))   # both hemispheres, far side
        a, b = lo.ravel(), la.ravel()
    elif src == 'radec':
        a, b = b0.xy2radec(*xy)
    elif src == 'km':
        a, b = b0.xy2km(*xy)
    else:
        a, b = b0.xy2angular(*xy)
    a = np.concatenate([a, [np.nan, 1.0, np.inf, -np.inf, 2.0]])
    b = np.concatenate([b, [1.0, np.nan, 3.0, 4.0, np.inf]])
    step = {'xy': 0.37, 'lonlat': 2.9, 'radec': 3e-6, 'km': 410.0, 'angular': 0.21}[src]
    k = np.arange(len(ser.bodies))[:, None]
    return (a, b), (a[None] + step * k, b[None] + 0.5 * step * k)


def _method_kwargs(groups, alt=0.0, nvn=None, nfn=None, pc=None, ang=None):
    kw = {}
    if 'alt' in groups:
        kw['alt'] = alt
    if 'nvn' in groups and nvn is not None:
        kw['not_visible_nan'] = nvn
    if 'nfn' in groups and nfn is not None:
        kw['not_found_nan'] = nfn
    if 'pc' in groups and pc is not None:
        kw['planetocentric'] = pc
    if 'ang' in groups and ang:
        kw.update(ang)
    return kw


def _series_kwargs(ser, name, kw):
    """series.transform's arguments for BodyXY method ``name`` called with ``kw``."""
    src, dst, _ = METHODS[name]
    out = dict(kw)
    if name == 'lonlat2xy' or (src == 'lonlat' and dst not in ('lonlat', 'centric')):
        out.setdefault('not_visible_nan', True)   # the BodyXY methods' default
    if name == 'centric2graphic_lonlat':
        out['planetocentric'] = True
    if src == 'km' and dst == 'angular':
        out['km2angular'] = ser.k2a
    return out


def _check(ser, name, per_frame, L, **opts):
    from planetmapper_b200 import series as S

    src, dst, groups = METHODS[name]
    kw = _method_kwargs(groups, **opts)
    shared, each = _inputs(ser, src)
    a, b = each if per_frame else shared
    before = L.launch_count()
    ga, gb = S.transform(ser.frames, src, dst, a, b, per_frame=per_frame, **_series_kwargs(ser, name, kw))
    launches = L.launch_count() - before
    ga, gb = ga.cpu().numpy(), gb.cpu().numpy()
    assert ga.shape == (len(ser.bodies),) + shared[0].shape
    for f, body in enumerate(ser.bodies):
        ra, rb = getattr(body, name)(*((a[f], b[f]) if per_frame else (a, b)), **kw)
        assert np.array_equal(ga[f], ra, equal_nan=True), (name, f, opts, per_frame)
        assert np.array_equal(gb[f], rb, equal_nan=True), (name, f, opts, per_frame)
    return ga, launches


@pytest.mark.parametrize('per_frame', [False, True])
@pytest.mark.parametrize('name', list(METHODS))
def test_every_method_matches_bodyxy_per_epoch(jupiter, name, per_frame):
    from planetmapper_b200 import _lib as L

    ga, launches = _check(jupiter, name, per_frame, L)
    assert launches == 1, launches   # one batched launch, not one per epoch
    assert np.isfinite(ga).any() and np.isnan(ga).any()   # hits and misses / hidden points / non-finite inputs
    if per_frame or name not in ('graphic2centric_lonlat', 'centric2graphic_lonlat'):   # these two are epoch-free
        assert not np.array_equal(ga[0], ga[-1], equal_nan=True)   # epochs differ


ALT_METHODS = [n for n, (_, _, g) in METHODS.items() if 'alt' in g]
PC_METHODS = [n for n, (_, _, g) in METHODS.items() if 'pc' in g]
NVN_METHODS = [n for n, (_, _, g) in METHODS.items() if 'nvn' in g]
ANG_METHODS = [n for n, (_, _, g) in METHODS.items() if 'ang' in g]


@pytest.mark.parametrize('alt', [750.0, -1200.0])
@pytest.mark.parametrize('name', ALT_METHODS)
def test_altitude(jupiter, name, alt):
    from planetmapper_b200 import _lib as L

    for per_frame in (False, True):
        _, launches = _check(jupiter, name, per_frame, L, alt=alt)
        assert launches == 1


@pytest.mark.parametrize('name', PC_METHODS)
def test_planetocentric(jupiter, name):
    from planetmapper_b200 import _lib as L

    for alt in (0.0, 900.0):
        _check(jupiter, name, True, L, pc=True, alt=alt)


@pytest.mark.parametrize('name', NVN_METHODS)
def test_not_visible_nan(jupiter, name):
    from planetmapper_b200 import _lib as L

    hidden_kept = _check(jupiter, name, False, L, nvn=False)[0]
    hidden_nan = _check(jupiter, name, False, L, nvn=True)[0]
    assert np.isnan(hidden_nan).sum() > np.isnan(hidden_kept).sum()
    _check(jupiter, name, True, L, nvn=True, alt=300.0)


@pytest.mark.parametrize('ang', [dict(origin_ra=None, origin_dec=None, coordinate_rotation=33.0),
                                 dict(origin_ra=None, origin_dec=None, coordinate_rotation=0.0),
                                 dict(origin_dec=-22.9),
                                 dict(origin_ra=5.6, origin_dec=22.7, coordinate_rotation=-140.0)])
@pytest.mark.parametrize('name', ANG_METHODS)
def test_custom_angular_frame(jupiter, name, ang):
    """origin_ra / origin_dec default to each epoch's own target RA / Dec; the km -> angular matrix is each
    epoch's (a single shared matrix would fail here)."""
    from planetmapper_b200 import _lib as L

    for per_frame in (False, True):
        _, launches = _check(jupiter, name, per_frame, L, ang=ang)
        assert launches == 1


NFN_METHODS = [n for n, (_, _, g) in METHODS.items() if 'nfn' in g]


def _from_xy(body, src, x, y):
    return (x, y) if src == 'xy' else getattr(body, f'xy2{src}')(x, y)


@pytest.mark.parametrize('name', NFN_METHODS)
def test_not_found_raises_exactly_when_some_epoch_misses(jupiter, name):
    from planetmapper_b200 import series as S
    from planetmapper_b200.body_xy import NotFoundError

    src, dst, _ = METHODS[name]
    ser = jupiter
    # the disc centre of every epoch, in the method's source system: a hit everywhere
    centre = [_from_xy(b, src, ser.x0[f], ser.y0[f]) for f, b in enumerate(ser.bodies)]
    a = np.array([[c[0]] * 3 for c in centre])
    b = np.array([[c[1]] * 3 for c in centre])
    a[:, 2], b[:, 2] = np.nan, np.nan   # a non-finite input is not a miss
    S.transform(ser.frames, src, dst, a, b, per_frame=True, not_found_nan=False)
    for body, ra, rb in zip(ser.bodies, a, b):
        getattr(body, name)(ra, rb, not_found_nan=False)
    # epochs 5 and 9 get one point in the sky
    sky = _from_xy(ser.bodies[0], src, -40.0, -40.0)
    for f in (5, 9):
        a[f, 1], b[f, 1] = sky
    with pytest.raises(NotFoundError, match=r'epoch 5\b'):
        S.transform(ser.frames, src, dst, a, b, per_frame=True, not_found_nan=False)
    for f, body in enumerate(ser.bodies):
        if f in (5, 9):
            with pytest.raises(NotFoundError):
                getattr(body, name)(a[f], b[f], not_found_nan=False)
        else:
            getattr(body, name)(a[f], b[f], not_found_nan=False)
    # shared points: one sky point misses at every epoch
    with pytest.raises(NotFoundError, match=r'epoch 0\b'):
        S.transform(ser.frames, src, dst, a[5], b[5], not_found_nan=False)
    got, _ = S.transform(ser.frames, src, dst, a, b, per_frame=True)   # not_found_nan=True: NaN, no error
    assert np.isnan(got.cpu().numpy()[[5, 9], 1]).all() and np.isfinite(got.cpu().numpy()[:, 0]).all()


def test_nonfinite_alt_follows_each_method(jupiter):
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import series as S

    ser = jupiter
    for name in ALT_METHODS:
        src, dst, _ = METHODS[name]
        shared, _ = _inputs(ser, src)
        kw = _series_kwargs(ser, name, {'alt': np.inf})
        try:
            getattr(ser.bodies[0], name)(*shared, alt=np.inf)
        except ValueError:
            with pytest.raises(ValueError):
                S.transform(ser.frames, src, dst, *shared, **kw)
            continue
        before = L.launch_count()
        ga, gb = S.transform(ser.frames, src, dst, *shared, **kw)
        assert L.launch_count() == before
        assert ga.shape == (len(ser.bodies),) + shared[0].shape and ga.isnan().all() and gb.isnan().all(), name


@pytest.mark.parametrize('name', ['xy2lonlat', 'lonlat2xy', 'xy2radec', 'km2lonlat', 'lonlat2angular',
                                  'graphic2centric_lonlat', 'centric2graphic_lonlat', 'km2angular'])
def test_europa_series(europa, name):
    """Triaxial target, analytic orbit (BASELINE config C5's Europa)."""
    from planetmapper_b200 import _lib as L

    groups = METHODS[name][2]
    for per_frame in (False, True):
        _check(europa, name, per_frame, L)
        if 'alt' in groups:
            _check(europa, name, per_frame, L, alt=35.0)
        if 'pc' in groups:
            _check(europa, name, per_frame, L, pc=True)
        if 'ang' in groups:
            _check(europa, name, per_frame, L, ang=dict(origin_dec=1.5, coordinate_rotation=12.0))


def test_scalar_and_grid_shapes(jupiter):
    from planetmapper_b200 import series as S

    ser = jupiter
    x, y = S.transform(ser.frames, 'lonlat', 'xy', 10.0, 20.0)
    assert tuple(x.shape) == (32,)
    for f, body in enumerate(ser.bodies):
        assert (x[f].item(), y[f].item()) == body.lonlat2xy(10.0, 20.0, not_visible_nan=False)
    lo, la = np.meshgrid(np.arange(0.0, 360, 45), np.arange(-60.0, 61, 30))
    x, y = S.transform(ser.frames, 'lonlat', 'xy', lo, la[:1])   # broadcast like the methods' inputs
    assert tuple(x.shape) == (32,) + lo.shape
    assert np.array_equal(x[7].cpu().numpy(), ser.bodies[7].lonlat2xy(lo, la[:1], not_visible_nan=False)[0],
                          equal_nan=True)
