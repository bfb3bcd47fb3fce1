#!/usr/bin/env python
"""Point transforms over a time series: one batched launch against a fresh BodyXY call per epoch (one GPU run):

    python tools/bench_series_points.py [--epochs 4096] [--points 10000] [--iters 20]
                                        [--out profiles/bench/series_points_b200.json]

Jupiter from Earth, one epoch a minute from 2005-01-01, each epoch with its own disc centre, radius and
rotation (build_series_frames with per-epoch arrays).  For ``lonlat2xy`` (a fixed grid of lon / lat points) and
``xy2radec`` (a fixed grid of pixels) it reports

- the device time of the batched kernel (CUDA events around --iters launches after warm-up, inputs already on
  the device): pm_lonlat2xy_batch / pm_transform_batch over all epochs x points;
- the host time of one ``series.transform`` call, numpy in, CUDA tensors out, ending in a device synchronise;
- the host time of the per-epoch loop over the same frames: ``BodyXY.set_disc_params`` + the method, numpy in,
  numpy out, for every epoch (BodyXY objects built beforehand; their constants are not timed);
- whether every row of the batched result equals the per-epoch call bit for bit;
- the GPU name and power limit, read in the same run.
The result is printed and written as JSON.
"""
import argparse
import json
import os
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


def device_ms(torch, fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / iters


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--epochs', type=int, default=4096)
    ap.add_argument('--points', type=int, default=10000)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bench', 'series_points_b200.json'))
    args = ap.parse_args()

    import torch

    import planetmapper_b200 as pm
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import frame as F
    from planetmapper_b200 import series as S

    if not torch.cuda.is_available():
        raise SystemExit('bench_series_points needs a CUDA device')
    prov = pm.get_default_provider()
    n, k = args.epochs, np.arange(args.epochs)
    ets = prov.utc2et('2005-01-01T00:00:00') + 60.0 * k   # inside the bundled ephemeris coverage
    nx = ny = 1024
    rot_deg = (15.0 + 0.01 * k) % 360.0
    disc = dict(x0=511.5 + 3.0 * np.sin(0.01 * k), y0=511.5 + 2.0 * np.cos(0.013 * k), r0=400.0 + 0.001 * k,
                rotation_radians=np.array([float(np.deg2rad(float(r))) % (2 * np.pi) for r in rot_deg]))
    t0 = time.perf_counter()
    frames = S.build_series_frames('Jupiter', ets, 'EARTH', nx=nx, ny=ny, **disc)
    t_frames = time.perf_counter() - t0
    S.shutdown_pool()
    side = int(round(args.points ** 0.5))
    lon, lat = np.meshgrid(np.linspace(0.0, 359.0, side), np.linspace(-80.0, 80.0, args.points // side))
    lon, lat = lon.ravel(), lat.ravel()
    xs, ys = np.meshgrid(np.linspace(50.0, 973.0, side), np.linspace(50.0, 973.0, args.points // side))
    xs, ys = xs.ravel(), ys.ravel()
    n_pts = lon.size

    bodies = []
    for f in range(n):
        body = pm.BodyXY(nx=nx, ny=ny, constants=F.build_body_constants(prov, 'Jupiter', None, 'EARTH',
                                                                          et=float(ets[f]), with_subsol=False))
        bodies.append(body)

    fd = L.to_device(frames)
    lo_d, la_d, x_d, y_d = (L.to_device(v) for v in (lon, lat, xs, ys))
    cases = {
        'lonlat2xy': (('lonlat', 'xy', lon, lat), dict(not_visible_nan=True),
                      lambda: L.lonlat2xy_batch(fd, lo_d, la_d, not_visible_nan=True), (lon, lat)),
        'xy2radec': (('xy', 'radec', xs, ys), {}, lambda: L.transform_batch(fd, 'xy', 'radec', x_d, y_d), (xs, ys)),
    }
    result = {'gpu': gpu_info(torch), 'epochs': n, 'points_per_epoch': n_pts, 'image': [nx, ny],
              'target': 'Jupiter from EARTH, one epoch every 60 s from 2005-01-01T00:00:00',
              'host_s_build_series_frames': t_frames, 'cases': {}}
    for name, (targs, kw, launch, (a, b)) in cases.items():
        ms = device_ms(torch, launch, args.iters)
        S.transform(frames, *targs, **kw)   # warm
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ga, gb = S.transform(frames, *targs, **kw)
        torch.cuda.synchronize()
        t_series = time.perf_counter() - t0
        ga, gb = ga.cpu().numpy(), gb.cpu().numpy()
        getattr(bodies[0], name)(a, b)   # warm
        per_epoch = []
        t0 = time.perf_counter()
        for f, body in enumerate(bodies):
            body.set_disc_params(disc['x0'][f], disc['y0'][f], disc['r0'][f], rot_deg[f])
            per_epoch.append(getattr(body, name)(a, b))
        t_loop = time.perf_counter() - t0
        identical = all(np.array_equal(ra, ga[f], equal_nan=True) and np.array_equal(rb, gb[f], equal_nan=True)
                        for f, (ra, rb) in enumerate(per_epoch))
        result['cases'][name] = {
            'device_ms_batched_kernel': ms,
            'points_per_s_batched_kernel': n * n_pts / (ms * 1e-3),
            'host_s_series_transform': t_series,
            'host_s_per_epoch_bodyxy_loop': t_loop,
            'host_ms_per_epoch_bodyxy_call': 1e3 * t_loop / n,
            'loop_over_series_transform': t_loop / t_series,
            'bit_identical_to_per_epoch_calls': bool(identical),
        }
    text = json.dumps(result, indent=1)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        fh.write(text + '\n')


if __name__ == '__main__':
    main()
