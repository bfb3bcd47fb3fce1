"""Times map_img's smoothing splines (spline_smoothing > 0) on the device against scipy on one CPU core.

Workloads:
  c4     a C4-shaped cube, 3000 planes of 64 x 64 (smooth field + 0.1 noise), s = m * 0.01 (the noise
         level: the knots grow part-way), degrees (3, 3); the map is 180 x 360 cells inside the image.
  large  one 1024 x 1024 plane, same recipe.  One plane keeps one CTA (one SM) busy, so this is the
         worst case for the device path.

Device times are host clocks around work that ends in a device synchronise, best of --repeat after a
warm-up: `fit` = pm_spline_prepare (NaN repair) + pm_regrid_fit + the ier copy (what map_img does before
its first cell), `gather` = pm_gather_regrid for every plane.  The CPU time is RectBivariateSpline on a
stated subsample of planes, one thread, scaled to the whole cube.  Prints one JSON object; --out writes it.

    python tools/bench_regrid.py [--planes 3000] [--cpu-sample 30] [--out FILE]

The B200 result is kept in profiles/bench/regrid_b200.json (its "gpu" field: card, power limit, max SM clock).
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


def cube_of(rng, n, ny, nx):
    yy, xx = np.mgrid[0:ny, 0:nx]
    a, b = rng.uniform(4, 12, n), rng.uniform(4, 12, n)
    return np.sin(xx[None] / a[:, None, None]) * np.cos(yy[None] / b[:, None, None]) + 0.1 * rng.normal(size=(n, ny, nx))


def device_times(L, torch, cube, s, xmap, ymap, repeat):
    dev = L.to_device(cube)
    xm, ym = L.to_device(xmap), L.to_device(ymap)

    def fit():
        return L.regrid_fit(dev, 3, 3, s)

    f = fit()
    L.gather_regrid(f, xm, ym)
    torch.cuda.synchronize()
    t_fit, t_gather = [], []
    for _ in range(repeat):
        t0 = time.perf_counter()
        f = fit()                                    # ends in the ier copy (a synchronise)
        t_fit.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        L.gather_regrid(f, xm, ym)
        torch.cuda.synchronize()
        t_gather.append(time.perf_counter() - t0)
    nxy = f.nxy.cpu().numpy()
    return min(t_fit), min(t_gather), f, nxy


def cpu_fit_time(cube, s, n_sample):
    from scipy.interpolate import RectBivariateSpline

    ny, nx = cube.shape[1:]
    t0 = time.perf_counter()
    knots = []
    for l in range(n_sample):
        r = RectBivariateSpline(np.arange(ny), np.arange(nx), cube[l], kx=3, ky=3, s=s)
        knots.append(tuple(len(t) for t in r.get_knots()))
    return (time.perf_counter() - t0) / n_sample, knots


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--planes', type=int, default=3000)
    ap.add_argument('--cpu-sample', type=int, default=30)
    ap.add_argument('--repeat', type=int, default=5)
    ap.add_argument('--out')
    args = ap.parse_args()
    import torch

    from planetmapper_b200 import _lib as L

    rng = np.random.default_rng(0)
    res = {'gpu': gpu_info(), 'torch': torch.__version__}
    # C4-shaped cube
    cube = cube_of(rng, args.planes, 64, 64)
    s = 64 * 64 * 0.01
    ym, xm = np.meshgrid(np.linspace(0.5, 62.5, 180), np.linspace(0.5, 62.5, 360), indexing='ij')
    t_fit, t_gather, fit, nxy = device_times(L, torch, cube, s, xm, ym, args.repeat)
    cpu_per_plane, knots = cpu_fit_time(cube, s, args.cpu_sample)
    assert [tuple(v) for v in nxy[:args.cpu_sample]] == knots, 'device and scipy knot counts differ'
    res['c4'] = {
        'planes': args.planes, 'shape': [64, 64], 's': s, 'degrees': [3, 3], 'map_cells': int(xm.size),
        'knots_x_mean': float(nxy[:, 0].mean()), 'knots_y_mean': float(nxy[:, 1].mean()),
        'knots_max': [int(nxy[:, 0].max()), int(nxy[:, 1].max())], 'knots_full': [64 + 4, 64 + 4],
        'device_fit_ms': 1e3 * t_fit, 'device_gather_ms': 1e3 * t_gather,
        'cpu_fit_ms_per_plane': 1e3 * cpu_per_plane, 'cpu_sample_planes': args.cpu_sample,
        'cpu_fit_ms_whole_cube_scaled': 1e3 * cpu_per_plane * args.planes,
        'fit_speedup_vs_one_core': cpu_per_plane * args.planes / t_fit,
    }
    # one large plane
    big = cube_of(rng, 1, 1024, 1024)
    s_big = 1024 * 1024 * 0.01
    ym, xm = np.meshgrid(np.linspace(0.5, 1022.5, 512), np.linspace(0.5, 1022.5, 1024), indexing='ij')
    t_fit, t_gather, fit, nxy = device_times(L, torch, big, s_big, xm, ym, max(1, args.repeat // 2))
    cpu_one, knots = cpu_fit_time(big, s_big, 1)
    assert tuple(nxy[0]) == knots[0], 'device and scipy knot counts differ (large plane)'
    res['large'] = {
        'shape': [1024, 1024], 's': s_big, 'degrees': [3, 3], 'knots': [int(v) for v in nxy[0]],
        'map_cells': int(xm.size), 'device_fit_ms': 1e3 * t_fit, 'device_gather_ms': 1e3 * t_gather,
        'cpu_fit_ms': 1e3 * cpu_one, 'fit_speedup_vs_one_core': cpu_one / t_fit,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(json.dumps(res, indent=2) + '\n')


if __name__ == '__main__':
    main()
