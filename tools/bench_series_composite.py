#!/usr/bin/env python
"""Composite of a mapped series: series.composite_mapped_series against iter_mapped_series plus a torch fold of its
output (one GPU run):

    python tools/bench_series_composite.py [--epochs 4096] [--out profiles/bench/series_composite_b200.json]

The unfused baseline is what a user writes without the composite: iterate iter_mapped_series, fetch every epoch's
EMISSION map (pm_backplanes_map_batch, one launch per batch) and fold each yielded (n, nλ) + grid tensor into
accumulators with torch ops, in epoch order (the mean's sum by plain adds, so linear agrees bit for bit).
Workload A: 32 Jupiter epochs x 512 planes x 64 x 64 onto the 0.25 deg grid (1440 x 720), linear and cubic, both
methods.  Cubic is a dense map there (253 cells per image pixel): the unfused path runs the DMMA gather, the
composite the scalar one, so they agree to 1e-12 relative instead of bit for bit.
Workload B: the --epochs Europa 1024 x 1024 series of bench_series_map.py's workload A onto the 1 deg grid,
min_emission with max_emission = 75, against the same baseline.
Device time: CUDA events around one call after a warm-up call of the same shape.  The bytes the unfused path moves
and the composite does not are computed from shapes: the gather's output (8 B per voxel-epoch) written once and read
back once by the fold.  The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_series_map import device_ms, gpu_info  # noqa: E402


def unfused(torch, L, S, frames, cubes, nx, ny, lons, lats, interp, method, max_emission, batch):
    """iter_mapped_series + per-batch EMISSION maps + a torch fold, in epoch order."""
    nl = 1 if cubes.dim() == 3 else cubes.shape[1]
    shape = (nl,) + lons.shape
    fd, lod, lad = L.to_device(frames), L.to_device(lons % 360), L.to_device(lats)
    emask = L.mask_from_names(['EMISSION'])
    need_e = method == 'min_emission' or max_emission is not None
    acc = torch.zeros(shape, dtype=torch.float64, device='cuda') if method == 'mean' else \
        torch.full(shape, float('nan'), dtype=torch.float64, device='cuda')
    tag = torch.zeros(shape, dtype=torch.int32, device='cuda') if method == 'mean' else \
        torch.full(shape, -1, dtype=torch.int32, device='cuda')
    key = torch.full(shape, float('inf'), dtype=torch.float64, device='cuda')
    cut = float('inf') if max_emission is None else max_emission
    for first, mapped in S.iter_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation=interp, batch=batch):
        n = mapped.shape[0]
        e = L.backplanes_map_batch(fd[first:first + n], lod, lad, emask)[:, 0] if need_e else None
        for k in range(n):
            v = mapped[k].reshape(shape)
            ok = ~torch.isnan(v)
            if need_e:
                ok &= (e[k] <= cut)
            if method == 'mean':
                acc = torch.where(ok, acc + v, acc)
                tag += ok
            else:
                better = ok & (e[k] < key)
                acc = torch.where(better, v, acc)
                key = torch.where(better, e[k], key)
                tag = torch.where(better, torch.full_like(tag, first + k), tag)
    if method == 'mean':
        acc = torch.where(tag > 0, acc / tag, torch.full_like(acc, float('nan')))
    return (acc[0], tag[0]) if cubes.dim() == 3 else (acc, tag)


def compare(torch, a, b, exact):
    (va, ta), (vb, tb) = a, b
    same_nan = bool(torch.equal(torch.isnan(va), torch.isnan(vb)))
    same_tag = bool(torch.equal(ta, tb))
    ok = ~torch.isnan(va)
    scale = float(vb[ok].abs().max()) if bool(ok.any()) else 1.0
    rel = float((va[ok] - vb[ok]).abs().max()) / scale if bool(ok.any()) else 0.0
    bitwise = bool(torch.equal(torch.nan_to_num(va, nan=0.0), torch.nan_to_num(vb, nan=0.0))) and same_nan
    agree = same_nan and same_tag and (bitwise if exact else rel <= 1e-12)
    return {'bit_identical': bitwise, 'nan_masks_equal': same_nan, 'tags_equal': same_tag, 'max_rel_diff': rel,
            'agree': agree}


def run_case(torch, L, S, frames, cubes, nx, ny, lons, lats, interp, method, cut, batch, exact):
    nl = 1 if cubes.dim() == 3 else cubes.shape[1]
    voxel_epochs = len(frames) * nl * lons.size
    fused = lambda: S.composite_mapped_series(frames, cubes, nx, ny, lons, lats, interpolation=interp, method=method,
                                              max_emission=cut, batch=batch)
    base = lambda: unfused(torch, L, S, frames, cubes, nx, ny, lons, lats, interp, method, cut, batch)
    res = {'interpolation': interp, 'method': method, 'max_emission': cut, 'batch': batch,
           'voxel_epochs': voxel_epochs}
    res['composite_ms'] = device_ms(torch, fused)
    res['unfused_ms'] = device_ms(torch, base)
    res['composite_voxel_epochs_per_s'] = voxel_epochs / (res['composite_ms'] * 1e-3)
    res['unfused_voxel_epochs_per_s'] = voxel_epochs / (res['unfused_ms'] * 1e-3)
    res['unfused_over_composite'] = res['unfused_ms'] / res['composite_ms']
    res['bytes_not_moved'] = {'gather_output_written': 8 * voxel_epochs, 'fold_reads_back': 8 * voxel_epochs}
    res['agreement'] = compare(torch, fused(), base(), exact)
    torch.cuda.empty_cache()
    return res


def workload_a(torch, pm, L, S):
    n_epochs, nl, sz = 32, 512, 64
    utcs = ['2005-01-01T0%d:%02d:00' % (h, m) for h in range(8) for m in (0, 15, 30, 45)][:n_epochs]
    prov = pm.get_default_provider()
    ets = np.array([prov.utc2et(u) for u in utcs])
    frames = S.build_series_frames('Jupiter', ets, 'EARTH', workers=1, nx=sz, ny=sz, x0=31.5, y0=31.5, r0=28.0)
    lo, la = np.meshgrid(np.arange(0.125, 360, 0.25)[::-1], np.arange(-89.875, 90, 0.25))
    gen = torch.Generator(device='cuda').manual_seed(1)
    cubes = torch.rand((n_epochs, nl, sz, sz), dtype=torch.float64, device='cuda', generator=gen)
    cubes[torch.rand(cubes.shape, device='cuda', generator=gen) < 0.01] = float('nan')
    res = {'workload': f'A: {n_epochs} Jupiter / EARTH epochs x {nl} planes x {sz}x{sz}, 0.25 deg rectangular grid '
                       f'({lo.shape[1]} x {lo.shape[0]})', 'cases': []}
    for interp in ('linear', 'cubic'):
        for method in ('mean', 'min_emission'):
            r = run_case(torch, L, S, frames, cubes, sz, sz, lo, la, interp, method, None, 8, interp == 'linear')
            print(json.dumps(r), flush=True)
            res['cases'].append(r)
    return res


def workload_b(torch, pm, L, S, n_epochs):
    sz = 1024
    prov = pm.get_default_provider()
    et_end = prov.utc2et('2005-01-01T00:00:00') - 3600.0
    ets = et_end - 60.0 * (n_epochs - 1 - np.arange(n_epochs))
    frames = S.build_series_frames('Europa', ets, 'EARTH', kepler=True, nx=sz, ny=sz, x0=(sz - 1) / 2,
                                   y0=(sz - 1) / 2, r0=0.45 * sz)
    S.shutdown_pool()
    lo, la = np.meshgrid(np.arange(0.5, 360, 1.0)[::-1], np.arange(-89.5, 90, 1.0))
    imgs = torch.empty((n_epochs, sz, sz), dtype=torch.float64, device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(0)
    for s in range(0, n_epochs, 128):
        part = torch.rand(imgs[s:s + 128].shape, dtype=torch.float64, device='cuda', generator=gen)
        part[torch.rand(part.shape, device='cuda', generator=gen) < 0.01] = float('nan')
        imgs[s:s + 128] = part
    del part
    res = {'workload': f'B: {n_epochs} Europa / EARTH epochs (analytic orbit), one {sz}x{sz} image each, 1 deg '
                       'rectangular grid (360 x 180), min_emission, max_emission 75', 'cases': []}
    for interp in ('linear', 'cubic'):
        r = run_case(torch, L, S, frames, imgs, sz, sz, lo, la, interp, 'min_emission', 75.0, 32, True)
        print(json.dumps(r), flush=True)
        res['cases'].append(r)
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--epochs', type=int, default=4096)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bench', 'series_composite_b200.json'))
    args = ap.parse_args()
    import torch

    import planetmapper_b200 as pm
    from planetmapper_b200 import _lib as L
    from planetmapper_b200 import series as S

    if not torch.cuda.is_available():
        raise SystemExit('bench_series_composite.py needs a CUDA device')
    gpu = gpu_info(torch)
    results = []
    for fn in (lambda: workload_a(torch, pm, L, S), lambda: workload_b(torch, pm, L, S, args.epochs)):
        r = fn()
        r['gpu'] = gpu
        results.append(r)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(results, f, indent=1)


if __name__ == '__main__':
    main()
