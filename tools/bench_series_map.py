#!/usr/bin/env python
"""Mapped time series: series.iter_mapped_series against the per-epoch paths (one GPU run):

    python tools/bench_series_map.py [--epochs 4096] [--out profiles/bench/series_map_b200.json]

Workload A (BASELINE config C5's shape, bench.py's bench_time_series setup): Europa from Earth (analytic orbit),
--epochs epochs 60 s apart, one 1024 x 1024 image per epoch (1 % NaN pixels, resident on the device), mapped
onto the 1 deg rectangular grid.  Timed with CUDA events after a warm-up of every timed shape:
- iter_mapped_series with nearest / linear / cubic, 32 epochs per batch and (cubic) the default batch;
- series.map_series with linear, 32 epochs per batch (the path that existed before);
- the same batches split into maps / prepare / gather (events around each launch group);
- the per-epoch loop a user needs for cubic without the series API: BodyXY.map_img(img, interpolation='cubic')
  on 64 epochs (bodies built beforehand), host time ending in a synchronise, scaled linearly to --epochs.
Workload B (a cube series): 32 epochs x 512 planes x 64 x 64 onto the 0.25 deg grid, nearest / linear / cubic:
the gather's output rate (8 B per mapped voxel) over gather kernel time, as a fraction of 7.7 TB/s, next to
Observation's gather of one epoch's cube (get_mapped_data_device's gather launch) of the same shape.
One JSON line per workload is printed; both go to --out with the GPU name and power limit read in the same run.
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

HBM_BYTES_PER_S = 7.7e12


def gpu_info(torch):
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['nvidia_smi'] = q
        parts = [p.strip() for p in q.split(',')]
        if len(parts) >= 2:
            info['power_limit'] = parts[1]
    except (OSError, subprocess.TimeoutExpired):
        info['nvidia_smi'] = None
    return info


def device_ms(torch, fn, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop)


def phases_ms(torch, L, S, frames_dev, cubes, nx, ny, lod, lad, mode, batch, nl):
    """Device time of the maps, the preparation and the gather of every batch of iter_mapped_series' loop."""
    stride = S._series_stride(nl, mode)
    n_frames = frames_dev.shape[0]
    xy = torch.empty((batch, 2) + tuple(lod.shape), dtype=torch.float64, device='cuda')
    out = torch.empty((batch, nl) + tuple(lod.shape), dtype=torch.float64, device='cuda')
    staged = None if stride == nl else torch.full((batch, stride, ny, nx), float('nan'), dtype=torch.float64,
                                                   device='cuda')
    mask = L.mask_from_names(['PIXEL-X', 'PIXEL-Y'])
    ev = []
    for first in range(0, n_frames, batch):
        n = min(batch, n_frames - first)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        L.backplanes_map_batch(frames_dev[first:first + n], lod, lad, mask, out=xy[:n])
        e[1].record()
        if staged is None:
            cube = cubes[first:first + n].reshape(n * nl, ny, nx)
        else:
            staged[:n, :nl].copy_(cubes[first:first + n].reshape(n, nl, ny, nx))
            cube = staged[:n].view(n * stride, ny, nx)
        src = cube if mode == L.INTERP_NEAREST else L.spline_prepare(cube, mode)
        e[2].record()
        L.gather_grouped(src, xy[:n, 0], xy[:n, 1], mode, nl, stride, out=out[:n])
        e[3].record()
        ev.append(e)
    torch.cuda.synchronize()
    return {'maps_ms': sum(e[0].elapsed_time(e[1]) for e in ev),
            'prepare_ms': sum(e[1].elapsed_time(e[2]) for e in ev),
            'gather_ms': sum(e[2].elapsed_time(e[3]) for e in ev)}


def workload_a(torch, pm, L, S, F, n_epochs):
    from planetmapper_b200.minispice.kepler import KeplerOrbitProvider

    sz = 1024
    prov = pm.get_default_provider()
    et_end = prov.utc2et('2005-01-01T00:00:00') - 3600.0
    ets = et_end - 60.0 * (n_epochs - 1 - np.arange(n_epochs))
    disc = dict(nx=sz, ny=sz, x0=(sz - 1) / 2, y0=(sz - 1) / 2, r0=0.45 * sz, rotation_radians=0.0)
    frames = S.build_series_frames('Europa', ets, 'EARTH', kepler=True, **disc)
    S.shutdown_pool()
    fd = L.to_device(frames)
    lo, la = np.meshgrid(np.arange(0.5, 360, 1.0)[::-1], np.arange(-89.5, 90, 1.0))
    lod, lad = L.to_device(lo % 360), L.to_device(la)
    imgs = torch.empty((n_epochs, sz, sz), dtype=torch.float64, device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(0)
    for s in range(0, n_epochs, 128):
        part = torch.rand(imgs[s:s + 128].shape, dtype=torch.float64, device='cuda', generator=gen)
        part[torch.rand(part.shape, device='cuda', generator=gen) < 0.01] = float('nan')
        imgs[s:s + 128] = part
    del part
    res = {'workload': f'A: {n_epochs} Europa / EARTH epochs (analytic orbit), one {sz}x{sz} image each, 1 deg '
                       'rectangular grid (360 x 180)', 'epochs': n_epochs}

    def run(interp, batch):
        for _ in S.iter_mapped_series(frames, imgs, sz, sz, lo, la, interpolation=interp, batch=batch):
            pass

    for interp in ('nearest', 'linear', 'cubic'):
        ms = device_ms(torch, lambda: run(interp, 32))
        res[f'iter_mapped_series_{interp}_batch32_ms'] = ms
        res[f'iter_mapped_series_{interp}_batch32_frames_per_s'] = n_epochs / ms * 1e3
        mode = {'nearest': L.INTERP_NEAREST, 'linear': L.INTERP_LINEAR, 'cubic': L.INTERP_CUBIC}[interp]
        res[f'iter_mapped_series_{interp}_batch32_split'] = phases_ms(torch, L, S, fd, imgs, sz, sz, lod, lad, mode,
                                                                      32, 1)
    ms = device_ms(torch, lambda: run('cubic', None))
    res['iter_mapped_series_cubic_default_batch_ms'] = ms
    res['iter_mapped_series_cubic_default_batch_frames_per_s'] = n_epochs / ms * 1e3
    mapped = torch.empty((n_epochs,) + lo.shape, dtype=torch.float64, device='cuda')
    ms = device_ms(torch, lambda: S.map_series(frames, imgs, sz, sz, lo, la, interpolation='linear', batch=32,
                                               out=mapped))
    res['map_series_linear_batch32_ms'] = ms
    res['map_series_linear_batch32_frames_per_s'] = n_epochs / ms * 1e3
    del mapped
    # the per-epoch loop: a BodyXY per epoch (built beforehand), map_img(cubic) of that epoch's image
    kp = KeplerOrbitProvider(prov)
    n_loop = min(64, n_epochs)
    bodies = []
    for k in range(n_loop):
        b = pm.BodyXY(constants=F.build_body_constants(kp, 'Europa', None, 'EARTH', et=float(ets[k])), nx=sz, ny=sz)
        b.set_disc_params(disc['x0'], disc['y0'], disc['r0'], 0.0)
        bodies.append(b)
    bodies[0].map_img(imgs[0], interpolation='cubic', degree_interval=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k, b in enumerate(bodies):
        b.map_img(imgs[k], interpolation='cubic', degree_interval=1)
    torch.cuda.synchronize()
    loop_s = time.perf_counter() - t0
    res['per_epoch_map_img_cubic_epochs_timed'] = n_loop
    res['per_epoch_map_img_cubic_s_per_epoch'] = loop_s / n_loop
    res['per_epoch_map_img_cubic_frames_per_s'] = n_loop / loop_s
    res['per_epoch_map_img_cubic_scaled_s'] = loop_s / n_loop * n_epochs
    res['per_epoch_note'] = (f'host time of {n_loop} BodyXY.map_img(cubic) calls (numpy out, bodies built '
                             f'beforehand) scaled linearly to {n_epochs} epochs')
    # the series equals the per-epoch result for the epochs timed
    first = next(iter(S.iter_mapped_series(frames[:4], imgs[:4], sz, sz, lo, la, interpolation='cubic')))[1]
    res['cubic_equals_map_img_first_4'] = all(
        np.array_equal(first[k].cpu().numpy(), bodies[k].map_img(imgs[k], interpolation='cubic', degree_interval=1),
                       equal_nan=True) for k in range(4))
    return res


def workload_b(torch, pm, L, S, F):
    n_epochs, nl, sz = 32, 512, 64
    utcs = ['2005-01-01T0%d:%02d:00' % (h, m) for h in range(8) for m in (0, 15, 30, 45)][:n_epochs]
    prov = pm.get_default_provider()
    ets = np.array([prov.utc2et(u) for u in utcs])
    disc = dict(nx=sz, ny=sz, x0=31.5, y0=31.5, r0=28.0, rotation_radians=0.0)
    frames = S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, **disc)
    lo, la = np.meshgrid(np.arange(0.125, 360, 0.25)[::-1], np.arange(-89.875, 90, 0.25))
    gen = torch.Generator(device='cuda').manual_seed(1)
    cubes = torch.rand((n_epochs, nl, sz, sz), dtype=torch.float64, device='cuda', generator=gen)
    cubes[torch.rand(cubes.shape, device='cuda', generator=gen) < 0.01] = float('nan')
    fd, lod, lad = L.to_device(frames), L.to_device(lo % 360), L.to_device(la)
    res = {'workload': f'B: {n_epochs} Jupiter / EARTH epochs x {nl} planes x {sz}x{sz}, 0.25 deg rectangular grid '
                       f'({lo.shape[1]} x {lo.shape[0]})', 'epochs': n_epochs, 'planes': nl}
    obs = pm.Observation(data=cubes[0].cpu().numpy(), target='Jupiter', utc=utcs[0], observer='EARTH')
    obs.set_disc_params(disc['x0'], disc['y0'], disc['r0'], 0.0)
    voxels_per_epoch = nl * lo.size
    for interp, mode in (('nearest', L.INTERP_NEAREST), ('linear', L.INTERP_LINEAR), ('cubic', L.INTERP_CUBIC)):
        batch = 8
        phases_ms(torch, L, S, fd, cubes, sz, sz, lod, lad, mode, batch, nl)   # warm-up
        split = phases_ms(torch, L, S, fd, cubes, sz, sz, lod, lad, mode, batch, nl)
        gbs = n_epochs * voxels_per_epoch * 8 / (split['gather_ms'] * 1e-3) / 1e9
        src = obs._map_source(obs._get_data_device(), interpolation=interp, degree_interval=0.25)
        buf = torch.empty((nl,) + lo.shape, dtype=torch.float64, device='cuda')
        single_ms = device_ms(torch, lambda: src.gather(0, nl, out=buf))
        single_gbs = voxels_per_epoch * 8 / (single_ms * 1e-3) / 1e9
        del buf, src
        res[interp] = dict(split, batch=batch, series_gather_gb_per_s=gbs, series_fraction_of_hbm=gbs * 1e9 / HBM_BYTES_PER_S,
                           single_cube_gather_ms=single_ms, single_cube_gather_gb_per_s=single_gbs,
                           single_cube_fraction_of_hbm=single_gbs * 1e9 / HBM_BYTES_PER_S,
                           series_over_single=gbs / single_gbs)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--epochs', type=int, default=4096)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bench', 'series_map_b200.json'))
    args = ap.parse_args()
    import torch

    import planetmapper_b200 as pm
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import frame as F
    from planetmapper_b200 import series as S

    if not torch.cuda.is_available():
        raise SystemExit('bench_series_map.py needs a CUDA device')
    gpu = gpu_info(torch)
    results = []
    for fn in (lambda: workload_a(torch, pm, L, S, F, args.epochs), lambda: workload_b(torch, pm, L, S, F)):
        r = fn()
        r['gpu'] = gpu
        print(json.dumps(r), flush=True)
        results.append(r)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(results, f, indent=1)


if __name__ == '__main__':
    main()
