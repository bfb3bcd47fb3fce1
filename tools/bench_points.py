#!/usr/bin/env python
"""Throughput of the per-point geometry queries of BodyXY (one GPU run):

    python tools/bench_points.py [--n-log2 24] [--iters 50] [--out profiles/bench/points_b200.json]

Jupiter from HST at 2005-01-01T00:00:00 (tests/golden/jupiter_hst_2005.json).  Reports

- device-timed points/s (CUDA events around --iters launches after warm-up) of the two kernels behind the methods
  on 2^n random points: pm_backplanes_map_host with the planes of illumination + azimuth + distance + radial
  velocity on lon / lat points uniform on the sphere, and pm_transform radec -> xy + pm_backplanes_points_host with
  the limb + ring planes on RA / Dec points within 3 equatorial radii of the body's centre;
- the end-to-end rate of the vectorised public methods, numpy in -> numpy out;
- the wall time of one scalar call of each public method (median of repeated calls);
- the GPU name and power limit, read in the same run.
The result is printed and written as JSON (default under profiles/bench/).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(torch):
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,power.max_limit', '--format=csv,noheader',
                            '-i', '0'], capture_output=True, text=True, timeout=30).stdout.strip()
        info['nvidia_smi'] = q
        parts = [p.strip() for p in q.split(',')]
        if len(parts) >= 2:
            info['power_limit'] = parts[1]
    except (OSError, subprocess.TimeoutExpired):
        info['nvidia_smi'] = None
    return info


def device_rate(torch, fn, n, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    stop.synchronize()
    ms = start.elapsed_time(stop) / iters
    return {'ms_per_launch_set': ms, 'points_per_s': n / (ms * 1e-3)}


def wall_rate(torch, fn, n, reps):
    fn()
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    return {'s_per_call': t, 'points_per_s': n / t}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--n-log2', type=int, default=24)
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bench', 'points_b200.json'))
    args = ap.parse_args()
    if args.iters < 50:
        ap.error('--iters must be at least 50')

    import torch

    import planetmapper_b200 as pm
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import frame as F

    with open(os.path.join(ROOT, 'tests', 'golden', 'jupiter_hst_2005.json')) as f:
        bc = F.BodyConstants.from_json_dict(json.load(f))
    body = pm.BodyXY(constants=bc)
    n = 1 << args.n_log2
    rng = np.random.default_rng(0)
    lon = rng.uniform(0.0, 360.0, n)
    lat = np.degrees(np.arcsin(rng.uniform(-1.0, 1.0, n)))       # uniform on the sphere
    r_eq_arcsec = body.target_diameter_arcsec / 2
    rho = 3.0 * r_eq_arcsec * np.sqrt(rng.uniform(0.0, 1.0, n))   # uniform on the disc of 3 equatorial radii
    phi = rng.uniform(0.0, 2 * np.pi, n)
    dec = body.target_dec + rho * np.sin(phi) / 3600.0
    ra = body.target_ra + rho * np.cos(phi) / 3600.0 / np.cos(np.radians(body.target_dec))

    result = {'gpu': gpu_info(torch), 'n_points': n, 'iters': args.iters,
              'target': 'Jupiter from HST, 2005-01-01T00:00:00'}
    fr = body._frame_host()
    lon_d, lat_d, ra_d, dec_d = (L.to_device(a) for a in (lon, lat, ra, dec))
    lonlat_mask = L.mask_from_names(['PHASE', 'INCIDENCE', 'EMISSION', 'AZIMUTH', 'DISTANCE', 'RADIAL-VELOCITY'])
    radec_mask = L.mask_from_names(['LIMB-LON-GRAPHIC', 'LIMB-LAT-GRAPHIC', 'LIMB-DISTANCE', 'RING-RADIUS',
                                    'RING-LON-GRAPHIC', 'RING-DISTANCE'])
    out_ll = torch.empty((L.popcount(lonlat_mask), n), dtype=torch.float64, device='cuda')
    out_rd = torch.empty((L.popcount(radec_mask), n), dtype=torch.float64, device='cuda')
    fd = body._frame_dev()

    def lonlat_kernels():
        L.backplanes_map_host(fr, lon_d, lat_d, lonlat_mask, out=out_ll)

    def radec_kernels():
        x, y, _ = L.transform(fd, 'radec', 'xy', ra_d, dec_d)
        L.backplanes_points_host(fr, x, y, radec_mask, out=out_rd)

    result['device'] = {
        'lonlat: pm_backplanes_map_host, illumination + azimuth + distance + radial velocity':
            device_rate(torch, lonlat_kernels, n, args.iters),
        'radec: pm_transform radec->xy + pm_backplanes_points_host, limb + ring':
            device_rate(torch, radec_kernels, n, args.iters),
    }
    e2e = {}
    for name, fn in (
            ('illumination_angles_from_lonlat', lambda: body.illumination_angles_from_lonlat(lon, lat)),
            ('azimuth_angle_from_lonlat', lambda: body.azimuth_angle_from_lonlat(lon, lat)),
            ('distance_from_lonlat', lambda: body.distance_from_lonlat(lon, lat)),
            ('radial_velocity_from_lonlat', lambda: body.radial_velocity_from_lonlat(lon, lat)),
            ('local_solar_time_from_lon', lambda: body.local_solar_time_from_lon(lon)),
            ('test_if_lonlat_visible', lambda: body.test_if_lonlat_visible(lon, lat)),
            ('limb_coordinates_from_radec', lambda: body.limb_coordinates_from_radec(ra, dec)),
            ('ring_plane_coordinates', lambda: body.ring_plane_coordinates(ra, dec))):
        e2e[name] = wall_rate(torch, fn, n, 5)
    result['end_to_end_numpy'] = e2e
    scalar = {}
    for name, fn in (
            ('illumination_angles_from_lonlat', lambda: body.illumination_angles_from_lonlat(153.0, -3.0)),
            ('azimuth_angle_from_lonlat', lambda: body.azimuth_angle_from_lonlat(153.0, -3.0)),
            ('local_solar_time_from_lon', lambda: body.local_solar_time_from_lon(153.0)),
            ('local_solar_time_string_from_lon', lambda: body.local_solar_time_string_from_lon(153.0)),
            ('distance_from_lonlat', lambda: body.distance_from_lonlat(153.0, -3.0)),
            ('radial_velocity_from_lonlat', lambda: body.radial_velocity_from_lonlat(153.0, -3.0)),
            ('test_if_lonlat_visible', lambda: body.test_if_lonlat_visible(153.0, -3.0)),
            ('limb_coordinates_from_radec', lambda: body.limb_coordinates_from_radec(196.3, -5.5)),
            ('ring_plane_coordinates', lambda: body.ring_plane_coordinates(196.3, -5.5))):
        scalar[name] = {'s_per_call': wall_rate(torch, fn, 1, 50)['s_per_call']}
    result['scalar_call'] = scalar
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == '__main__':
    main()
