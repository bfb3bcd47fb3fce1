"""
Referee of the point transforms (pm_transform, pm_xy2lonlat, pm_lonlat2xy and their _batch forms, which every
coordinate method of Body / BodyXY, test_if_lonlat_visible and series.transform run through) against the oracle
evaluated in 80-bit arithmetic, on the random geometries of the image referee
(test_host_check.py::test_device_code_random_geometries_vs_extended_precision), the close observer and the
OTHER_BODIES frames.

Every one of the 20 pairs, with not_visible_nan on and off, planetocentric lon / lat, custom angular frames and
altitudes scaled to the body, is evaluated three times: by the kernels' code (host build or device), by the FP64
oracle and by the oracle in long double (the driver below links the same rewritten source as build_ld_oracle).
The kernel code must be as close to the 80-bit result as the FP64 oracle is, over EVERY point both find - limb,
poles and grazing emission included - and its NaN masks and miss counts must equal the 80-bit ones except at
points within 1e-9 of a decision (ray tangency, emission = 90 deg, equal light times of the ray cast).

Points are not drawn only where things are easy: a third of the xy / sky points sit within 2 px of the limb (a few
just outside it), and the lon / lat points include a band of emission 80 - 100 deg around the visibility limit.
"""
import ctypes
import itertools
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import OTHER_BODIES, PID, angle_diff, close_observer_constants, img_case, random_geometry_parts
from planetmapper_b200 import frame as F

SYSTEMS = ['xy', 'angular', 'km', 'radec', 'lonlat']
PAIRS = [(s, d) for s, d in itertools.product(SYSTEMS, SYSTEMS) if s != d]
COORD = {'xy': 0, 'angular': 1, 'km': 2, 'radec': 3, 'lonlat': 4}
N_POINTS = 1024          # per job (a pair and variant on one geometry), the same on every geometry
GRAZING = 1e-9           # 80-bit distance to a decision below which a NaN flip is waived (and counted)
# bars of _tolerance (test_transforms.py) floor the referee's denominators; xy: 1e-9 of the frame
FLOOR = {'angular': 2e-8, 'km': 1e-4, 'radec': 1e-12, 'lonlat': 1e-9}
RATIO_MAX, RATIO_RMS = 10.0, 3.0


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


# ---------------------------------------------------------------------------------
# 80-bit runner: pmo_transform of the long-double oracle, many jobs per process, plus each point's distance to
# the decision its NaN mask depends on
# ---------------------------------------------------------------------------------
TRANSFORM_DRV = r"""
#include <stdio.h>
#include <stdlib.h>
#include "pm_oracle_ld.c"

typedef long double LD;

/* How far (80-bit) a point is from flipping between found and NaN: the tangency margin of the ray (scaled
 * radii) for a lon / lat destination; for a lon / lat source with not_visible_nan, the emission angle's distance
 * to 90 deg (radians) on the surface, or above / below it the ray cast's tangency margin and light-time
 * difference (in body radii).  INFINITY where nothing is decided. */
static LD grazing_margin(const PMFrame *f, const LD *aux, int src, int dst, LD a, LD b, LD alt, uint32_t flags) {
    LD ov[3], p[3], lt, m = NAN;
    if (!(isfinite(a) && isfinite(b))) return INFINITY;
    if (dst == PM_COORD_LONLAT || dst == PM_COORD_CENTRIC) {
        if (src == PM_COORD_LONLAT) return INFINITY;
        if (src == PM_COORD_RADEC) radec_deg2obsvec_norm(a, b, ov);
        else if (src == PM_COORD_ANGULAR) angular2obsvec_m(aux, a, b, ov);
        else if (src == PM_COORD_KM) angular2obsvec_m(f->M, aux[9] * a + aux[10] * b, aux[11] * a + aux[12] * b, ov);
        else xy2obsvec_norm(f, a, b, ov);
        if (!finite3(ov)) return INFINITY;
        sincpt(f, ov, p, &lt, &m);
        return fabs(m);
    }
    if (src != PM_COORD_LONLAT || !(flags & PM_FLAG_NOT_VISIBLE_NAN)) return INFINITY;
    LD lo, la, tv[3];
    lonlat2obsvec(f, a, b, alt, flags & ~PM_FLAG_NOT_VISIBLE_NAN, ov, &lo, &la, tv);
    if (alt == 0) {
        PointState s;
        point_state(f, tv, f->lt0, 1, &s);
        return fabs(s.emissn - HALFPI);
    }
    if (!sincpt(f, ov, p, &lt, &m)) return fabs(m);
    PointState si, sp;
    point_state(f, p, f->lt0, 0, &si);
    point_state(f, tv, f->lt0, 0, &sp);
    return fmin(fabs(m), fabs(sp.lt - si.lt) * f->clight / f->radii[0]);
}

/* argv[1]: n_jobs, then per job src, dst, alt, flags, n, the frame, aux13, a[n], b[n] (doubles);
 * argv[2] receives per job n_missed, out_a[n], out_b[n], margin[n], rounded to double at the very end */
int main(int argc, char **argv) {
    FILE *fp = fopen(argv[1], "rb");
    if (!fp) return 1;
    fseek(fp, 0, SEEK_END);
    long sz = ftell(fp);
    rewind(fp);
    double *in = malloc(sz);
    if (fread(in, 1, sz, fp) != (size_t)sz) return 1;
    fclose(fp);
    int64_t nj = (int64_t)in[0], ip = 1, op = 0;
    int64_t *ioff = malloc(8 * nj), *ooff = malloc(8 * nj);
    for (int64_t j = 0; j < nj; j++) {
        int64_t n = (int64_t)in[ip + 4];
        ioff[j] = ip;
        ooff[j] = op;
        ip += 5 + PM_FRAME_NDOUBLES + 13 + 2 * n;
        op += 1 + 3 * n;
    }
    double *out = malloc(8 * op);
#pragma omp parallel for schedule(dynamic)
    for (int64_t j = 0; j < nj; j++) {
        const double *h = in + ioff[j];
        const int src = (int)h[0], dst = (int)h[1];
        const LD alt = h[2];
        const uint32_t flags = (uint32_t)h[3];
        const int64_t n = (int64_t)h[4];
        PMFrame f;
        LD *fl = (LD *)&f, aux[13];
        for (int i = 0; i < PM_FRAME_NDOUBLES; i++) fl[i] = h[5 + i];
        for (int i = 0; i < 13; i++) aux[i] = h[5 + PM_FRAME_NDOUBLES + i];
        const double *a = h + 5 + PM_FRAME_NDOUBLES + 13, *b = a + n;
        LD *la = malloc(sizeof(LD) * 4 * n), *lb = la + n, *oa = lb + n, *ob = oa + n;
        for (int64_t i = 0; i < n; i++) { la[i] = a[i]; lb[i] = b[i]; }
        int64_t missed = 0;
        pmo_transform(&f, src, dst, la, lb, n, alt, flags, aux, oa, ob, &missed);
        double *o = out + ooff[j];
        o[0] = (double)missed;
        for (int64_t i = 0; i < n; i++) {
            o[1 + i] = (double)oa[i];
            o[1 + n + i] = (double)ob[i];
            o[1 + 2 * n + i] = (double)grazing_margin(&f, aux, src, dst, la[i], lb[i], alt, flags);
        }
        free(la);
    }
    fp = fopen(argv[2], "wb");
    if (!fp || fwrite(out, 8, op, fp) != (size_t)op) return 2;
    fclose(fp);
    return 0;
}
"""


def build_ld_transform(bdir):
    """Compiles TRANSFORM_DRV against the 80-bit oracle in `bdir`; returns run(jobs) -> [(a, b, n_missed, margin)]."""
    from test_host_check import write_ld_sources

    write_ld_sources(bdir)
    exe = os.path.join(bdir, 'transform_ld')
    open(os.path.join(bdir, 'drv_transform.c'), 'w').write(TRANSFORM_DRV)
    subprocess.run(['gcc', '-O2', '-w', '-fopenmp', '-o', exe, 'drv_transform.c', '-lm'], cwd=bdir, check=True,
                   capture_output=True)

    def run(jobs):
        parts = [np.array([len(jobs)], dtype=np.float64)]
        for j in jobs:
            parts += [np.array([COORD[j['src']], COORD[j['dst']], j['alt'], j['flags'], j['a'].size], dtype=np.float64),
                      j['frame'], j['aux'], j['a'], j['b']]
        fin, fout = os.path.join(bdir, 'jobs.bin'), os.path.join(bdir, 'out.bin')
        np.concatenate(parts).tofile(fin)
        subprocess.run([exe, fin, fout], check=True)
        out = np.fromfile(fout)
        res, k = [], 0
        for j in jobs:
            n = j['a'].size
            res.append((out[k + 1:k + 1 + n], out[k + 1 + n:k + 1 + 2 * n], int(out[k]), out[k + 1 + 2 * n:k + 1 + 3 * n]))
            k += 1 + 3 * n
        return res
    return run


# ---------------------------------------------------------------------------------
# Geometries, points and jobs
# ---------------------------------------------------------------------------------
def _geometries():
    """(label, constants, (nx, ny, x0, y0, r0, rotation)) of the 48 random geometries, the close observer and
    the OTHER_BODIES frames."""
    import planetmapper_b200 as pm

    out = []
    for seed in range(48):
        bc, disc, _, label = random_geometry_parts(seed)
        out.append((label.rsplit(' alt=', 1)[0], bc, disc))   # altitudes here are the variants'
    out.append(('Jupiter from Amalthea', close_observer_constants(), (120, 90, 61.0, 40.5, 55.0, 200.0)))
    for target, observer, *disc in OTHER_BODIES:
        bc = F.build_body_constants(pm.get_default_provider(), target, '2004-12-31T00:00:00', observer)
        out.append((f'{target}/{observer}', bc, tuple(disc)))
    return out


def _aux(bc, custom):
    """aux13 of pm_transform: the obsvec -> angular matrix (the target's own, or a frame with its origin offset
    and turned by 33 deg), then the km -> angular matrix."""
    if custom:
        m = F.obsvec2angular_matrix(bc.target_ra + 0.002, bc.target_dec - 0.001, 33.0)
    else:
        m = F.obsvec2angular_matrix(bc.target_ra, bc.target_dec, 0.0)
    return np.concatenate([m.ravel(), F.km2angular_matrix(bc).ravel()])


def _limb_xy(oracle, fr, x0, y0, r0, rng, k):
    """k points on the limb in pixels: radial bisection on hit / miss of the FP64 oracle from the disc centre."""
    th = rng.uniform(0, 2 * np.pi, k)
    c, s = np.cos(th), np.sin(th)
    lo, hi = np.zeros(k), np.full(k, 1.5 * r0 + 2.0)
    assert np.all(np.isnan(oracle.xy2lonlat(fr, x0 + hi * c, y0 + hi * s)[0]))
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        hit = np.isfinite(oracle.xy2lonlat(fr, x0 + mid * c, y0 + mid * s)[0])
        lo, hi = np.where(hit, mid, lo), np.where(hit, hi, mid)
    return lo, c, s


def _xy_points(oracle, fr, disc, rng, n):
    """60 % uniform over the frame, 30 % within 2 px of the limb, 10 % just outside it (1e-7 .. 1e-2 px)."""
    nx, ny, x0, y0, r0, _ = disc
    nu, nb = int(0.6 * n), int(0.3 * n)
    nj = n - nu - nb
    rho, c, s = _limb_xy(oracle, fr, x0, y0, r0, rng, nb + nj)
    d = np.concatenate([rng.uniform(-2, 2, nb), 10 ** rng.uniform(-7, -2, nj)])
    x = np.concatenate([rng.uniform(-0.5, nx - 0.5, nu), x0 + (rho + d) * c])
    y = np.concatenate([rng.uniform(-0.5, ny - 0.5, nu), y0 + (rho + d) * s])
    return x, y


def _lonlat_points(oracle, fr, rng, n):
    """Uniform on the sphere (cos-lat weighted), lon in [-360, 720); 40 % with emission 80 - 100 deg."""
    lon, lat = rng.uniform(-360, 720, 40 * n), np.rad2deg(np.arcsin(rng.uniform(-1, 1, 40 * n)))
    emi = oracle.backplanes_map(fr, lon, lat, mask=1 << PID['EMISSION'])[0]
    band = np.flatnonzero((emi >= 80) & (emi <= 100))[:int(0.4 * n)]
    rest = np.setdiff1d(np.arange(lon.size), band)[:n - band.size]
    sel = np.concatenate([band, rest])
    return lon[sel], lat[sel]


SPECIALS = (np.array([np.nan, 1.0, np.inf, -np.inf]), np.array([1.0, np.nan, 1.0, 0.5]))


def _with_specials(a, b):
    a, b = a.copy(), b.copy()
    a[:4], b[:4] = SPECIALS
    return np.ascontiguousarray(a), np.ascontiguousarray(b)


def _variants(src, dst):
    """The variants of test_transforms._compare_pair with altitudes scaled to the body (fractions of its largest
    radius).  Below the surface a point is always hidden with not_visible_nan, so the negative altitude runs
    with it off; at +0.5 r points are seen past the limb."""
    if src == 'lonlat':
        vs = [dict(nvn=True), dict(nvn=False), dict(nvn=True, alt=0.02), dict(nvn=True, alt=0.5),
              dict(nvn=False, alt=-0.005), dict(nvn=True, pc=True), dict(nvn=True, pc=True, alt=0.02),
              dict(nvn=False, pc=True, alt=-0.005)]
    elif dst == 'lonlat':
        vs = [dict(), dict(alt=0.02), dict(alt=0.5), dict(alt=-0.005), dict(pc=True), dict(pc=True, alt=0.02)]
    else:
        vs = [dict()]
    if 'angular' in (src, dst):
        vs = [dict(v, custom=c) for v in vs for c in (False, True)]
    return vs


def _vkey(v):
    parts = [k for k in ('nvn', 'pc', 'custom') if v.get(k)]
    if v.get('alt'):
        parts.append(f'alt={v["alt"]:+g}r')
    return ' '.join(parts) or 'plain'


def _make_jobs(oracle):
    jobs = []
    for gi, (label, bc, disc) in enumerate(_geometries()):
        rng = np.random.default_rng(7000 + gi)
        r = float(np.max(bc.radii))
        fr0 = img_case(bc, *disc)
        aux = {c: _aux(bc, c) for c in (False, True)}
        pts = {'xy': _with_specials(*_xy_points(oracle, fr0, disc, rng, N_POINTS)),
               'lonlat': _with_specials(*_lonlat_points(oracle, fr0, rng, N_POINTS))}
        for sky in ('radec', 'km', 'angular'):
            for c in ((False, True) if sky == 'angular' else (False,)):
                x, y = _xy_points(oracle, fr0, disc, rng, N_POINTS)
                pts[sky, c] = _with_specials(*oracle.transform(fr0, 'xy', sky, x, y, aux13=aux[c])[:2])
        frames = {}
        for src, dst in PAIRS:
            for v in _variants(src, dst):
                alt = v.get('alt', 0.0) * r
                key = alt if dst == 'lonlat' else 0.0
                if key not in frames:
                    frames[key] = np.ascontiguousarray(img_case(bc, *disc, alt=key), dtype=np.float64)
                a, b = pts[src] if src in ('xy', 'lonlat') else pts[src, v.get('custom', False) and src == 'angular']
                jobs.append(dict(geometry=gi, label=label, pair=(src, dst), vkey=_vkey(v), src=src, dst=dst,
                                 frame=frames[key], nxy=max(disc[0], disc[1]), alt=alt,
                                 flags=(1 if v.get('nvn') else 0) | (4 if v.get('pc') else 0),
                                 aux=aux[v.get('custom', False)], a=a, b=b))
    return jobs


@pytest.fixture(scope='module')
def referee_jobs(oracle, tmp_path_factory):
    """Every job with its 80-bit result ('exact': a, b, n_missed, margin) and FP64 oracle result ('fp64')."""
    if not shutil.which('gcc'):
        pytest.skip('gcc not available')
    jobs = _make_jobs(oracle)
    run = build_ld_transform(str(tmp_path_factory.mktemp('transform_ld')))   # always rebuilt from the current source
    for j, ex in zip(jobs, run(jobs)):
        j['exact'] = ex
        j['fp64'] = oracle.transform(j['frame'], j['src'], j['dst'], j['a'], j['b'], alt=j['alt'],
                                     not_visible_nan=bool(j['flags'] & 1), planetocentric=bool(j['flags'] & 4),
                                     aux13=j['aux'])
    return jobs


# ---------------------------------------------------------------------------------
# The referee rule
# ---------------------------------------------------------------------------------
def _errors(dst, a, b, xa, xb):
    """Per output coordinate |got - exact|; longitudes (and RA) through angle_diff and cos(lat)."""
    if dst in ('lonlat', 'radec'):
        with np.errstate(invalid='ignore'):
            return angle_diff(a, xa) * np.cos(np.deg2rad(xb)), np.abs(b - xb)
    return np.abs(a - xa), np.abs(b - xb)


def referee(job, ga, gb, gm):
    """Returns (failure messages, stats) of one evaluation (ga, gb, gm) of `job` against its 80-bit result: NaN
    masks and n_missed equal outside grazing points, and per coordinate kernel-vs-80-bit <= 3x oracle-vs-80-bit
    in rms, <= 10x in the maximum, over every point all three evaluations find."""
    xa, xb, xm, margin = job['exact']
    oa, ob, _ = job['fp64']
    grazing = margin < GRAZING
    mism = (np.isnan(ga) != np.isnan(xa)) | (np.isnan(gb) != np.isnan(xb))
    fails = []
    n_bad = int((mism & ~grazing).sum())
    if n_bad:
        i = int(np.flatnonzero(mism & ~grazing)[0])
        fails.append(f'{n_bad} NaN-mask mismatches outside grazing points, e.g. ({job["a"][i]!r}, {job["b"][i]!r}): '
                     f'got ({ga[i]}, {gb[i]}), 80-bit ({xa[i]}, {xb[i]}), margin {margin[i]:.2e}')
    flips = [f'({job["a"][i]!r}, {job["b"][i]!r}) margin {margin[i]:.1e}: got ({ga[i]:.6g}, {gb[i]:.6g}), 80-bit '
             f'({xa[i]:.6g}, {xb[i]:.6g})' for i in np.flatnonzero(mism & grazing)]
    n_flip = len(flips)
    if abs(gm - xm) > n_flip:
        fails.append(f'n_missed {gm}, 80-bit {xm} ({n_flip} grazing flips)')
    both = np.isfinite(ga) & np.isfinite(gb) & np.isfinite(xa) & np.isfinite(xb) & np.isfinite(oa) & \
        np.isfinite(ob) & ~grazing
    if both.sum() < 50:
        fails.append(f'only {int(both.sum())} points compared')
    floor = 1e-9 * job['nxy'] if job['dst'] == 'xy' else FLOOR[job['dst']]
    stats = dict(n_grazing=int(grazing.sum()), flips=flips, r_max=0.0, r_rms=0.0, d_max=0.0, o_max=0.0)
    de2 = _errors(job['dst'], ga, gb, xa, xb)
    oe2 = _errors(job['dst'], oa, ob, xa, xb)
    for coord, de, oe in zip('ab', de2, oe2):
        de, oe = de[both], oe[both]
        if not de.size:
            continue
        r_max = float(de.max() / max(oe.max(), floor))
        r_rms = float(np.sqrt(np.mean(de ** 2)) / max(np.sqrt(np.mean(oe ** 2)), 0.1 * floor))
        stats['r_max'], stats['r_rms'] = max(stats['r_max'], r_max), max(stats['r_rms'], r_rms)
        stats['d_max'], stats['o_max'] = max(stats['d_max'], float(de.max())), max(stats['o_max'], float(oe.max()))
        if r_max > RATIO_MAX or r_rms > RATIO_RMS:
            fails.append(f'{coord}-coordinate: kernel-vs-80-bit / oracle-vs-80-bit = '
                         f'{r_max:.2f} (max), {r_rms:.2f} (rms); max errors {de.max():.3e} / {oe.max():.3e}')
    return fails, stats


class Report:
    """Per (entry point, pair, variant) over every geometry: worst ratios, largest errors, grazing points."""

    def __init__(self):
        self.rows, self.fails, self.flips = {}, [], []

    def add(self, entry, job, ga, gb, gm):
        fails, st = referee(job, ga, gb, gm)
        key = (entry, f'{job["src"]}->{job["dst"]}', job['vkey'])
        row = self.rows.setdefault(key, dict(r_max=0.0, r_rms=0.0, d_max=0.0, o_max=0.0, n_grazing=0, n_flip=0))
        for k in ('r_max', 'r_rms', 'd_max', 'o_max'):
            row[k] = max(row[k], st[k])
        row['n_grazing'] += st['n_grazing']
        row['n_flip'] += len(st['flips'])
        where = f'{entry} {key[1]} [{key[2]}] {job["label"]}'
        self.flips += [f'{where}: {m}' for m in st['flips']]
        self.fails += [f'{where}: {m}' for m in fails]

    def finish(self):
        print(f'\n{"entry":<12} {"pair":<16} {"variant":<26} {"ratio max":>9} {"ratio rms":>9} {"max err":>10} '
              f'{"oracle err":>10} {"grazing":>7} {"flips":>5}')
        for (entry, pair, vkey), r in sorted(self.rows.items()):
            print(f'{entry:<12} {pair:<16} {vkey:<26} {r["r_max"]:9.2f} {r["r_rms"]:9.2f} {r["d_max"]:10.2e} '
                  f'{r["o_max"]:10.2e} {r["n_grazing"]:7d} {r["n_flip"]:5d}')
        print('NaN flips at grazing points (80-bit margin < %g), waived:' % GRAZING, *self.flips or ['none'], sep='\n  ')
        assert not self.fails, f'{len(self.fails)} failures:\n' + '\n'.join(self.fails[:30])


# ---------------------------------------------------------------------------------
# Host build of the kernels' code
# ---------------------------------------------------------------------------------
def _is_xy2lonlat(job):
    return job['pair'] == ('xy', 'lonlat') and not job['flags'] & 4


@pytest.mark.parametrize('src,dst', PAIRS)
def test_host_transforms_vs_extended_precision(HC, referee_jobs, src, dst):
    rep = Report()
    for j in (j for j in referee_jobs if j['pair'] == (src, dst)):
        a, b, n = j['a'], j['b'], j['a'].size
        oa, ob, missed = np.empty(n), np.empty(n), ctypes.c_int64(0)
        assert HC.hc_transform(_p(j['frame']), ctypes.c_int(COORD[src]), ctypes.c_int(COORD[dst]), _p(a), _p(b),
                               ctypes.c_int64(n), ctypes.c_double(j['alt']), ctypes.c_uint32(j['flags']), _p(j['aux']),
                               _p(oa), _p(ob), ctypes.byref(missed)) == 0
        rep.add('transform', j, oa, ob, missed.value)
        if _is_xy2lonlat(j):
            assert HC.hc_xy2lonlat(_p(j['frame']), _p(a), _p(b), ctypes.c_int64(n), _p(oa), _p(ob),
                                   ctypes.byref(missed)) == 0
            rep.add('xy2lonlat', j, oa, ob, missed.value)
        if (src, dst) == ('lonlat', 'xy'):
            assert HC.hc_lonlat2xy(_p(j['frame']), _p(a), _p(b), ctypes.c_int64(n), ctypes.c_double(j['alt']),
                                   ctypes.c_uint32(j['flags']), _p(oa), _p(ob)) == 0
            rep.add('lonlat2xy', j, oa, ob, j['exact'][2])
    rep.finish()


# ---------------------------------------------------------------------------------
# Device
# ---------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def L():
    import torch

    from planetmapper_b200 import _lib

    assert torch.cuda.is_available()
    _lib.load_library()
    return _lib


def _device_single(L, j):
    """The single-frame launches of one job: {entry: (a, b, n_missed)} as numpy."""
    d = L.to_device
    fr, a, b = d(j['frame']), d(j['a']), d(j['b'])
    oa, ob, m = L.transform(fr, j['src'], j['dst'], a, b, alt=j['alt'], not_visible_nan=bool(j['flags'] & 1),
                            planetocentric=bool(j['flags'] & 4), aux13=j['aux'])
    out = {'transform': (oa.cpu().numpy(), ob.cpu().numpy(), int(m.item()))}
    if _is_xy2lonlat(j):
        lon, lat, m = L.xy2lonlat(fr, a, b)
        out['xy2lonlat'] = (lon.cpu().numpy(), lat.cpu().numpy(), int(m.item()))
    if j['pair'] == ('lonlat', 'xy'):
        x, y = L.lonlat2xy(fr, a, b, bool(j['flags'] & 1), alt=j['alt'], planetocentric=bool(j['flags'] & 4))
        out['lonlat2xy'] = (x.cpu().numpy(), y.cpu().numpy(), j['exact'][2])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('src,dst', PAIRS)
def test_device_transforms_vs_extended_precision(L, referee_jobs, src, dst):
    rep = Report()
    for j in (j for j in referee_jobs if j['pair'] == (src, dst)):
        for entry, (oa, ob, m) in _device_single(L, j).items():
            rep.add(entry, j, oa, ob, m)
    rep.finish()


@pytest.mark.gpu
@pytest.mark.parametrize('src,dst', PAIRS)
def test_mixed_body_batches_equal_single_frame_launches(L, referee_jobs, src, dst):
    """Every geometry of a pair and variant - different bodies, frames and angular tables - in ONE
    transform_batch / xy2lonlat_batch / lonlat2xy_batch launch with per-frame points: each row equals its
    single-frame launch bit for bit, n_missed included.  A launch takes one altitude (km), so altitude variants
    run every row at the first row's altitude, and so do the single-frame launches they are compared with."""
    groups = {}
    for j in referee_jobs:
        if j['pair'] == (src, dst):
            groups.setdefault(j['vkey'], []).append(j)
    for vkey, js in groups.items():
        assert len(set(j['geometry'] for j in js)) == len(js) > 50
        alt, flags = js[0]['alt'], js[0]['flags']
        js = [dict(j, alt=alt) for j in js]
        frames = L.to_device(np.stack([j['frame'] for j in js]))
        a, b = L.to_device(np.stack([j['a'] for j in js])), L.to_device(np.stack([j['b'] for j in js]))
        oa, ob, m = L.transform_batch(frames, src, dst, a, b, per_frame=True, alt=alt, not_visible_nan=bool(flags & 1),
                                      planetocentric=bool(flags & 4),
                                      aux13_dev=L.to_device(np.stack([j['aux'] for j in js])))
        got = {'transform': (oa.cpu().numpy(), ob.cpu().numpy(), m.cpu().numpy())}
        if _is_xy2lonlat(js[0]):
            lon, lat, m = L.xy2lonlat_batch(frames, a, b, per_frame=True)
            got['xy2lonlat'] = (lon.cpu().numpy(), lat.cpu().numpy(), m.cpu().numpy())
        if (src, dst) == ('lonlat', 'xy'):
            x, y = L.lonlat2xy_batch(frames, a, b, per_frame=True, not_visible_nan=bool(flags & 1), alt=alt,
                                     planetocentric=bool(flags & 4))
            got['lonlat2xy'] = (x.cpu().numpy(), y.cpu().numpy(), None)
        for r, j in enumerate(js):
            single = _device_single(L, j)
            for entry, (ga, gb, gm) in got.items():
                sa, sb, sm = single[entry]
                where = f'{entry} {src}->{dst} [{vkey}] row {r}: {j["label"]}'
                assert np.array_equal(ga[r], sa, equal_nan=True) and np.array_equal(gb[r], sb, equal_nan=True), where
                if gm is not None:
                    assert int(gm[r]) == sm, where


# ---------------------------------------------------------------------------------
# Image-kernel instantiations on the same geometries
# ---------------------------------------------------------------------------------
DEFAULT_STACK = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LOCAL-SOLAR-TIME', 'LON-CENTRIC', 'LAT-CENTRIC', 'PHASE', 'INCIDENCE',
                 'EMISSION', 'AZIMUTH', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER']
SURFACE_SUBSET = ['LAT-GRAPHIC', 'LON-CENTRIC', 'EMISSION', 'RADIAL-VELOCITY']


@pytest.mark.gpu
def test_image_kernel_instantiations_on_random_geometries(L):
    """The default 12-plane stack (backplanes_img_param_kernel<false, kDefaultStackMask, *>) and a surface-only
    subset (<false, 0, *>) - what BodyXY's surface-plane calls launch, on triaxial bodies the non-spin-symmetric
    instantiations - equal the ALL_PLANES slots bit for bit on every geometry; and all geometries in ONE
    pm_backplanes_img launch, which picks the spin-symmetric path per CTA, equal the single-frame launches."""
    geoms = _geometries()
    assert sum('Europa' in label for label, _, _ in geoms) >= 3    # triaxial: spin_sym off
    stacks = [L.mask_from_names(DEFAULT_STACK), L.mask_from_names(SURFACE_SUBSET)]
    batch_frames = []
    for seed in range(48):
        bc, disc, alt, label = random_geometry_parts(seed)
        nx, ny = disc[:2]
        fr = img_case(bc, *disc, alt)
        full = L.backplanes_img_host(fr, nx, ny).cpu().numpy()
        for mask in stacks:
            ids = [k for k in range(len(L.PLANE_NAMES)) if mask >> k & 1]
            sub = L.backplanes_img_host(fr, nx, ny, mask).cpu().numpy()
            assert np.array_equal(sub, full[ids], equal_nan=True), (label, [L.PLANE_NAMES[k] for k in ids])
        s = 64.0 / max(nx, ny)
        batch_frames.append(img_case(bc, 64, 64, disc[2] * s, disc[3] * s, disc[4] * s, disc[5], alt))
    for label, bc, disc in geoms[48:]:
        s = 64.0 / max(disc[:2])
        batch_frames.append(img_case(bc, 64, 64, disc[2] * s, disc[3] * s, disc[4] * s, disc[5]))
    frames = np.stack(batch_frames)
    for mask in [L.ALL_PLANES] + stacks:
        batch = L.backplanes_img(L.to_device(frames), 64, 64, mask).cpu().numpy()
        for k, fr in enumerate(frames):
            one = L.backplanes_img_host(fr, 64, 64, mask).cpu().numpy()
            assert np.array_equal(batch[k], one, equal_nan=True), (k, hex(mask))
            assert np.isfinite(one[0]).sum() > 10, k
