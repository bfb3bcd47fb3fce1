#!/usr/bin/env python
"""
bench.py - headline benchmark of the B200-native PlanetMapper hot path.

    python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K --warmup W   (CPU reference arm)

Metric (BASELINE.json): full-backplane Mpix/s (FP64) + mapped-cube voxels/s.
Workload at every N (weak scaling, no data-path collective): each rank computes the
12-plane default backplane stack of one Jupiter/HST 2048 x 2048 frame per step
(BASELINE.json configs[1], "C2").  `value` is the whole-job Mpix/s of the kernel (CUDA events; the
92 frame constants ride in the launch as a kernel parameter, nothing else is read); `e2e` is the same
metric through the drop-in public call - a fresh BodyXY and `get_backplane_img(name)` for each of the
12 names, host arrays out - with the device -> host copies inside the timed region, next to the raw
pinned-copy ceiling of the same bytes measured in the same run.
`mapped_cube` reports configs[3] ("C4": 3000 x 64 x 64 cube -> 0.1 deg grid, 6.48 M cells, nearest /
linear / cubic) in voxels/s: device-resident (wavelength planes sharded over the ranks, chunked because the
155.5 GB output does not fit next to its own copy) and end to end through
`Observation.iter_mapped_data` (double-buffered pinned staging).

The reference (pure Python + spiceypy) cannot be installed here or on the GPU box (no spiceypy / CSPICE
wheels, no network), so `--impl reference` and `cpu_baseline` time the CPU restatement in oracle/
(kind "port": C + OpenMP for the geometry, the REAL scipy for the map resampling) on the box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2_NAMES = ['LON-GRAPHIC', 'LAT-GRAPHIC', 'LON-CENTRIC', 'LAT-CENTRIC', 'INCIDENCE', 'EMISSION', 'PHASE',
            'AZIMUTH', 'LOCAL-SOLAR-TIME', 'DISTANCE', 'RADIAL-VELOCITY', 'DOPPLER']
METRIC = 'full-backplane Mpix/s (FP64) + mapped-cube voxels/s at 1-8 B200 vs host CPU'
SZ = 2048
CPU_SAMPLE_SZ = 2048
# the SAME string in both arms (the driver compares them)
WORKLOAD = ('C2: Jupiter/HST 2005-01-01T00:00:00, one 2048x2048 frame per GPU per step, 12-plane default backplane '
            'stack (' + ', '.join(C2_NAMES) + '), disc centred, r0 = 0.9 (n-1)/2')
C4_NL, C4_SZ, C4_CHUNK = 3000, 64, 512


def load_bc():
    from planetmapper_b200 import frame as F

    with open(os.path.join(ROOT, 'tests', 'golden', 'jupiter_hst_2005.json')) as f:
        return F.BodyConstants.from_json_dict(json.load(f))


def c2_frame(bc, sz=SZ):
    from planetmapper_b200 import frame as F

    c = (sz - 1) / 2
    return F.pack_frame(bc, nx=sz, ny=sz, x0=c, y0=c, r0=0.9 * c, rotation_radians=0.0)


def plane_mask(names):
    from planetmapper_b200 import _lib as L

    return L.mask_from_names(names)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    QUERY = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
             'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits', '-lms', '100',
                 '-i', str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for n, v in zip(names, parts[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'power_w_max': max(power) if power else None, 'samples': len(sm), 'reasons': sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured (MEASURED_PEAKS.json)'
    return {'hbm_gbs': 6650.0}, 'fallback (B200_PROFILING.md)'


def algorithmic_flops_per_frame(planes_host, frame):
    """FP64 flops of one C2 launch = per-class flop counts (profiles/flops_per_pixel.json:
    2 DFMA + DMUL + DADD this kernel executes per on-disc / in-circle-miss / outside pixel,
    measured with ncu thread-instruction counters by tools/count_flops_ncu.py) x the number
    of pixels of each class in the timed frame."""
    from planetmapper_b200 import frame as F

    path = os.path.join(ROOT, 'profiles', 'flops_per_pixel.json')
    with open(path) as f:
        fpp = json.load(f)
    nx, ny = int(F.frame_field(frame, 'nx')[0]), int(F.frame_field(frame, 'ny')[0])
    x0, y0 = F.frame_field(frame, 'x0')[0], F.frame_field(frame, 'y0')[0]
    r_cut2 = F.frame_field(frame, 'r_cut2')[0]
    yy, xx = np.mgrid[0:ny, 0:nx]
    in_circle = ((xx - x0) ** 2 + (yy - y0) ** 2) <= r_cut2
    on_disc = np.isfinite(planes_host)
    n_on = int(on_disc.sum())
    n_miss = int((in_circle & ~on_disc).sum())
    n_out = int((~in_circle).sum())
    c = fpp['c2_12plane']
    flops = n_on * c['on_disc'] + n_miss * c['in_circle_miss'] + n_out * c['outside_circle']
    det = fpp.get('detail', {})
    counts = {'on_disc': n_on, 'in_circle_miss': n_miss, 'outside_circle': n_out}
    warp_inst = {k: sum(counts[c_] * det[c_][k] for c_ in counts) for k in ('warp_inst', 'fp64_pipe_inst')} if det else None
    return flops, {'on_disc_px': n_on, 'in_circle_miss_px': n_miss, 'outside_px': n_out,
                   'flops_per_px': c, 'flop_definition': fpp['flop_definition'], 'warp_instructions': warp_inst}


# share of the FP64 instructions of the C2 kernel that are DFMAs with three distinct register sources
# (static property of the build: ncu source page of profiles/, 12.94 M of 51.85 M warp instructions)
THREE_REGISTER_DFMA_SHARE = 0.25


def issue_model(classes, ms, clocks, sms):
    """Issue cycles of one launch by the rules measured with tools/microbench/fp64_operands.cu (an FP64
    instruction holds the sub-partition's issue port 2 cycles, 3 with three register sources; every other
    instruction costs 0.5 ... 1 cycle) over the sub-partition cycles the launch took."""
    wi = classes.get('warp_instructions')
    mhz = (clocks or {}).get('sm_mhz')
    if not wi or not mhz:
        return None
    fp64, other = wi['fp64_pipe_inst'], wi['warp_inst'] - wi['fp64_pipe_inst']
    fp64_cycles = fp64 * (2.0 + THREE_REGISTER_DFMA_SHARE)
    elapsed = ms * 1e-3 * mhz * 1e6 * sms * 4
    return {'fp64_warp_inst': fp64, 'other_warp_inst': other, 'three_register_dfma_share': THREE_REGISTER_DFMA_SHARE,
            'issue_cycles_fp64': fp64_cycles, 'issue_cycles_total_lo_hi': [fp64_cycles + 0.5 * other, fp64_cycles + other],
            'elapsed_subpartition_cycles': elapsed,
            'frac_lo_hi': [(fp64_cycles + 0.5 * other) / elapsed, (fp64_cycles + other) / elapsed],
            'what': 'warp instructions = per-class counts of profiles/flops_per_pixel.json x the pixels of each class; '
                    'cycles per instruction from profiles/r2_fp64_operands.log (DESIGN.md 3.4)'}


def ncu_summary(key):
    """Counters of the committed ncu capture of this kernel (profiles/ncu_summary.json,
    written by tools/ncu_summary.py from the .ncu-rep files of the same commands)."""
    path = os.path.join(ROOT, 'profiles', 'ncu_summary.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(key)
    return None


def ncu_traffic(key):
    s = ncu_summary(key)
    return None if not s else s.get('dram_bytes_per_launch')


def cpu_port_mpix(sz, repeats=1):
    """Times the CPU oracle (C port of the reference path) on a sz x sz C2-like frame."""
    from oracle import oracle as O

    O.build()
    bc = load_bc()
    fr = c2_frame(bc, sz)
    mask = plane_mask(C2_NAMES)
    O.backplanes_img(fr, 32, 32, mask)  # load + warm
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        O.backplanes_img(fr, sz, sz, mask)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return sz * sz / best / 1e6, best


def omp_threads():
    n = os.environ.get('OMP_NUM_THREADS')
    if n:
        return int(n)
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_one_core_mpix():
    """The same port on ONE core: a child process with OMP_NUM_THREADS=1 (the OpenMP runtime reads it at
    load) on the C2 geometry at 1024 x 1024 (same disc fraction, a quarter of the pixels)."""
    env = dict(os.environ, OMP_NUM_THREADS='1')
    out = subprocess.run([sys.executable, os.path.abspath(__file__), '--cpu-child', '1024'], env=env,
                         capture_output=True, text=True, timeout=600)
    return float(out.stdout.strip().splitlines()[-1])


def c4_inputs(n_planes=C4_NL):
    """C4's synthetic cube and grid (SURVEY 8(d)): default_rng(0) normal(1, 0.1), 1 % NaN pixels, plane 17 all NaN."""
    rng = np.random.default_rng(0)
    cube = rng.normal(1.0, 0.1, (n_planes, C4_SZ, C4_SZ))
    cube[rng.random((n_planes, C4_SZ, C4_SZ)) < 0.01] = np.nan
    if n_planes > 17:
        cube[17] = np.nan
    lons = np.arange(0.05, 360, 0.1)[::-1]
    lats = np.arange(-90 + 0.05, 90, 0.1)
    lo, la = np.meshgrid(lons, lats)
    return cube, lo, la


def c4_frame(bc):
    from planetmapper_b200 import frame as F

    return F.pack_frame(bc, nx=C4_SZ, ny=C4_SZ, x0=31.5, y0=31.5, r0=28.0, rotation_radians=0.0)


def cpu_baselines_extra(bc):
    """BASELINE.md section 3: CPU rows for the other configs, each on a bounded sample.
    C4 uses the REAL scipy (RectBivariateSpline.ev etc. arranged as BodyXY.map_img arranges them,
    oracle/map_img_oracle.py) on the first 8 planes at the full 0.1 deg grid - scipy is single threaded, the
    reference loops planes serially, cost is linear in planes; the x / y maps (C oracle, all threads) are
    timed separately because the reference computes them once per cube.  C3 / C5: the C port."""
    import planetmapper_b200 as pm
    from oracle import map_img_oracle as MO
    from oracle import oracle as O
    from planetmapper_b200 import frame as F

    res = {}
    n_s = 8
    cube, lo, la = c4_inputs(24)
    fr = c4_frame(bc)
    xy_mask = plane_mask(['PIXEL-X', 'PIXEL-Y'])
    t0 = time.perf_counter()
    xy = O.backplanes_map(fr, lo, la, xy_mask)
    t_xy = time.perf_counter() - t0
    c4 = {'sample': f'planes 16..{16 + n_s - 1} of the C4 cube (incl. the all-NaN plane 17) at the full 0.1 deg grid '
                    f'({lo.size} cells), real scipy, 1 core; x / y maps by the C port on {omp_threads()} threads',
          'xy_map_s': t_xy, 'xy_map_mcells_per_s': lo.size / t_xy / 1e6, 'unit': 'voxels/s', 'cores': 1, 'kind': 'port',
          'note': 'numpy bookkeeping around the same scipy calls (map_cube_fast, checked equal to the line-by-line '
                  'form of BodyXY.map_img); the reference itself walks every cell in a Python loop and is slower still'}
    for interp in ('nearest', 'linear', 'cubic'):
        t0 = time.perf_counter()
        MO.map_cube_fast(cube[16:16 + n_s], xy[0], xy[1], interp)
        dt = time.perf_counter() - t0
        c4[interp] = {'voxels_per_s': n_s * lo.size / dt, 's_per_plane': dt / n_s,
                      'whole_cube_s_extrapolated': dt / n_s * C4_NL + t_xy}
    res['mapped_cube'] = c4
    # C3: Saturn 4096 x 4096, ring planes + DISTANCE, the full frame
    bcs = F.build_body_constants(pm.get_default_provider(), 'Saturn', '2004-12-30T12:00:00', 'EARTH')
    sz = 4096
    frs = F.pack_frame(bcs, nx=sz, ny=sz, x0=(sz - 1) / 2, y0=(sz - 1) / 2, r0=800.0, rotation_radians=0.0)
    m3 = plane_mask(['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE', 'DISTANCE'])
    t0 = time.perf_counter()
    O.backplanes_img(frs, sz, sz, m3)
    dt = time.perf_counter() - t0
    res['saturn_rings'] = {'img_mpix_per_s': sz * sz / dt / 1e6, 's': dt, 'cores': omp_threads(), 'kind': 'port',
                           'sample': 'the full C3 frame (4096 x 4096, 3 ring planes + DISTANCE)'}
    # C5: 4 frames of the Europa series at 1024 x 1024, 12-plane stack (constants + pixels)
    from planetmapper_b200 import series as S

    prov = pm.get_default_provider()
    et_end = prov.utc2et('2005-01-01T00:00:00') - 3600.0
    ets = et_end - 60.0 * np.arange(4)
    sz = 1024
    t0 = time.perf_counter()
    frames = S.build_series_frames('Europa', ets, 'EARTH', nx=sz, ny=sz, x0=(sz - 1) / 2, y0=(sz - 1) / 2, r0=0.45 * sz,
                                   workers=1, kepler=True)
    t_host = time.perf_counter() - t0
    m5 = plane_mask(C2_NAMES)
    t0 = time.perf_counter()
    for fr5 in frames:
        O.backplanes_img(fr5, sz, sz, m5)
    dt = time.perf_counter() - t0
    res['time_series'] = {'backplanes_mpix_per_s': len(frames) * sz * sz / dt / 1e6, 'cores': omp_threads(), 'kind': 'port',
                          'host_constants_ms_per_frame': t_host / len(frames) * 1e3,
                          'sample': '4 of the 4096 Europa frames (1024 x 1024, 12-plane stack)',
                          'whole_series_s_extrapolated': dt / len(frames) * 4096}
    return res


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return 0
    # all the host threads this process may use (torchrun pins OMP_NUM_THREADS=1 for its workers);
    # set before the OpenMP runtime of the oracle library is loaded
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    os.environ['OMP_NUM_THREADS'] = str(cores)
    from oracle import oracle as O

    O.build()
    bc = load_bc()
    fr = c2_frame(bc, CPU_SAMPLE_SZ)
    mask = plane_mask(C2_NAMES)
    for _ in range(max(args.warmup, 1)):
        O.backplanes_img(fr, CPU_SAMPLE_SZ, CPU_SAMPLE_SZ, mask)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.backplanes_img(fr, CPU_SAMPLE_SZ, CPU_SAMPLE_SZ, mask)
    dt = (time.perf_counter() - t0) / args.steps
    value = CPU_SAMPLE_SZ * CPU_SAMPLE_SZ / dt / 1e6
    sample = (f'one full C2 frame ({CPU_SAMPLE_SZ}x{CPU_SAMPLE_SZ}, 12-plane stack) per step, OpenMP over pixels')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'Mpix/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'sample': sample},
        'cpu_baseline': {'value': value, 'unit': 'Mpix/s', 'cores': omp_threads(), 'kind': 'port',
                         'sample': sample,
                         'note': 'reference (Python + spiceypy/CSPICE) is not installable here; this is the '
                                 'C restatement in oracle/, far faster than the reference itself'},
        'e2e': {'value': value, 'unit': 'Mpix/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))
    return 0


def bench_mapped_cube(L, torch, pm, bc, rank, world, e2e=True):
    """C4: 3000 x 64 x 64 cube -> 0.1 deg rectangular grid.  Wavelength planes are sharded over the ranks in
    plane quads (strong scaling: rank r maps planes lo..hi of the 3000), device resident in chunks of 512
    planes; then the same shard end to end through Observation.iter_mapped_data (linear)."""
    from planetmapper_b200.shard import max_over_ranks, shard_range

    sz, nl_total, chunk = C4_SZ, C4_NL, C4_CHUNK
    q_lo, q_hi = shard_range(nl_total // 4, rank, world)
    lo_p, hi_p = 4 * q_lo, 4 * q_hi
    fr = c4_frame(bc)
    cube_h, lo, la = c4_inputs()
    fd = L.to_device(fr)
    lod, lad = L.to_device(lo), L.to_device(la)
    xy_mask = L.mask_from_names(['PIXEL-X', 'PIXEL-Y'])
    xy = L.backplanes_map(fd, lod, lad, xy_mask)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    xy = L.backplanes_map(fd, lod, lad, xy_mask)
    e1.record()
    torch.cuda.synchronize()
    xy_ms = e0.elapsed_time(e1)
    cube = L.to_device(cube_h[lo_p:hi_p])     # this rank's planes only: NaN repair / spline fit shard with the gather
    n_cells = lo.size
    out = torch.empty((chunk,) + lo.shape, dtype=torch.float64, device='cuda')
    res = {'workload': 'C4: 3000x64x64 cube (1% NaN px, one all-NaN plane) -> 0.1 deg grid '
                       f'({lo.shape[1]}x{lo.shape[0]} = {n_cells} cells), planes sharded over {world} rank(s) '
                       f'(this rank: {lo_p}..{hi_p}), chunks of {chunk} planes into a reused device buffer '
                       '(full output 155.5 GB)',
           'scaling': 'strong', 'planes_this_rank': hi_p - lo_p,
           'xy_map_ms': xy_ms, 'unit': 'voxels/s', 'visible_cell_fraction': float(torch.isfinite(xy[0]).double().mean())}
    peaks, src = measured_peaks()
    for mode, name in ((L.INTERP_NEAREST, 'nearest'), (L.INTERP_LINEAR, 'linear'), (L.INTERP_CUBIC, 'cubic')):
        def one_pass():
            prep_ms = 0.0
            if mode == L.INTERP_NEAREST:
                src_ = cube
            else:
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                src_ = L.spline_prepare(cube, mode)
                p1.record()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            n_launch = 0
            for s_ in range(0, hi_p - lo_p, chunk):
                n = min(chunk, hi_p - lo_p - s_)
                L.gather(src_, xy[0], xy[1], mode, plane_begin=s_, plane_count=n, out=out[:n])
                n_launch += 1
            g1.record()
            torch.cuda.synchronize()
            if mode != L.INTERP_NEAREST:
                prep_ms = p0.elapsed_time(p1)
            return g0.elapsed_time(g1), prep_ms, n_launch
        one_pass()
        gather_ms, prep_ms, n_launch = one_pass()
        vox_rank = (hi_p - lo_p) * n_cells
        alg_bytes = 8.0 * vox_rank + 8.0 * (hi_p - lo_p) * sz * sz + 16.0 * n_cells * n_launch
        total_ms = max_over_ranks(gather_ms + prep_ms, world, device='cuda')
        res[name] = {
            'voxels_per_s': nl_total * n_cells / (total_ms * 1e-3), 'ms_all_ranks': total_ms,
            'gather_ms': gather_ms, 'prepare_ms': prep_ms, 'launches': n_launch,
            'roofline': {'bound': 'hbm', 'achieved': alg_bytes / (gather_ms * 1e-3) / 1e9,
                         'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                         'frac': alg_bytes / (gather_ms * 1e-3) / 1e9 / peaks['hbm_gbs'], 'peak_source': src,
                         'traffic': ncu_traffic(f'gather_{name}'),
                         'traffic_note': 'ncu dram bytes of ONE launch of this kernel at the bench chunk (512 planes)',
                         'algorithmic_bytes_per_voxel': alg_bytes / vox_rank},
        }
    del out
    if e2e:
        # end to end: the public streaming call on this rank's planes, host arrays out (pinned double buffer),
        # D2H inside the timed region; the consumer touches one value per plane
        obs = pm.Observation(data=cube_h[lo_p:hi_p], constants=bc)
        obs.set_disc_params(31.5, 31.5, 28.0, 0.0)
        per = 32

        first_chunk_s = [None]

        def stream():
            acc, n_planes = 0.0, 0
            t_start = time.perf_counter()
            for first, mapped in obs.iter_mapped_data('linear', planes_per_chunk=per, degree_interval=0.1):
                if first_chunk_s[0] is None:
                    first_chunk_s[0] = time.perf_counter() - t_start
                acc += float(np.nansum(mapped[:, 900, 1800]))
                n_planes += mapped.shape[0]
            return acc, n_planes
        # warm: one short pass builds the x / y maps, the spline operand and the pinned buffers
        warm = pm.Observation(data=cube_h[lo_p:lo_p + 2 * per], constants=bc)
        warm.set_disc_params(31.5, 31.5, 28.0, 0.0)
        for _ in warm.iter_mapped_data('linear', planes_per_chunk=per, degree_interval=0.1):
            pass
        del warm
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        t0 = time.perf_counter()
        acc, n_planes = stream()
        torch.cuda.synchronize()
        dt = max_over_ranks((time.perf_counter() - t0) * 1e3, world, device='cuda')
        nbytes = n_planes * n_cells * 8
        res['e2e_linear'] = {
            'api': "Observation(data=cube[lo:hi]).iter_mapped_data('linear', degree_interval=0.1): x / y maps, NaN "
                   'repair, gather in 32-plane chunks, each chunk to pinned host memory while the next is gathered',
            'voxels_per_s': nl_total * n_cells / (dt * 1e-3), 'ms_all_ranks': dt, 'planes_this_rank': n_planes,
            'd2h_bytes_this_rank': int(nbytes), 'd2h_gb_per_s_this_rank': nbytes / (dt * 1e-3) / 1e9,
            'setup_s_until_first_chunk': first_chunk_s[0],
            'setup_what': 'lon / lat grid on the host, x / y maps, cube upload, NaN repair, staging buffers, first chunk',
            'stream_gb_per_s_after_setup': (nbytes * (1 - per / max(n_planes, per))) / max(dt * 1e-3 - first_chunk_s[0], 1e-9) / 1e9,
            'h2d_bytes_this_rank': int(cube_h[lo_p:hi_p].nbytes), 'checksum': acc}
        del obs
    if world > 1:
        # result assembly (SURVEY 8(e)): 64 mapped planes of every rank into one device buffer on rank 0,
        # NCCL point-to-point straight into the destination slices (GPU-to-GPU over NVLink)
        import torch.distributed as dist

        from planetmapper_b200.shard import gather_blocks

        per = 64
        blk = torch.empty((per,) + lo.shape, dtype=torch.float64, device='cuda')
        L.gather(cube, xy[0], xy[1], L.INTERP_NEAREST, plane_begin=0, plane_count=per, out=blk)
        whole = torch.empty((per * world,) + lo.shape, dtype=torch.float64, device='cuda') if rank == 0 else None
        for timed in (False, True):
            dist.barrier()
            torch.cuda.synchronize()
            e0.record()
            gather_blocks(blk, per * world, world, rank, dst=0, out=whole)
            e1.record()
            torch.cuda.synchronize()
            dist.barrier()
        nbytes = per * (world - 1) * n_cells * 8
        res['assemble_on_rank0'] = {'planes_per_rank': per, 'bytes_received': nbytes, 'ms': e0.elapsed_time(e1),
                                    'gb_per_s': nbytes / e0.elapsed_time(e1) / 1e6,
                                    'how': 'NCCL send / irecv into slices of one buffer (shard.gather_blocks)'}
        del whole, blk
    return res


def bench_saturn_rings(L, torch, pm):
    """C3: Saturn 4096 x 4096 with the ring planes, plus orthographic and azimuthal-equal-area
    backplane maps (size 2048).  Saturn from EARTH 12 h before the end of the bundled SPK
    (SURVEY 8(d)); r0 = 800 px so the A ring (2.27 r_eq) is in frame."""
    from planetmapper_b200 import frame as F

    bc = F.build_body_constants(pm.get_default_provider(), 'Saturn', '2004-12-30T12:00:00', 'EARTH')
    sz, r0 = 4096, 800.0
    fr = F.pack_frame(bc, nx=sz, ny=sz, x0=(sz - 1) / 2, y0=(sz - 1) / 2, r0=r0, rotation_radians=0.0)
    names = ['RING-RADIUS', 'RING-LON-GRAPHIC', 'RING-DISTANCE', 'DISTANCE']
    mask = L.mask_from_names(names)
    fd = L.to_device(fr[None])
    out = torch.empty((1, len(names), sz, sz), dtype=torch.float64, device='cuda')

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    img_ms = timed(lambda: L.backplanes_img(fd, sz, sz, mask, out=out))
    ring_px = int(torch.isfinite(out[0, names.index('RING-RADIUS')]).sum())
    res = {'workload': f'C3: Saturn / EARTH 2004-12-30T12:00, {sz}x{sz}, r0 = {r0:.0f} px, planes ' + ', '.join(names),
           'img_ms': img_ms, 'img_mpix_per_s': sz * sz / img_ms / 1e3, 'ring_plane_px': ring_px}
    size = 2048
    c = np.linspace(-1.01 * max(1.0, bc.r_polar / bc.r_eq), 1.01 * max(1.0, bc.r_polar / bc.r_eq), size)
    for kind, name in ((L.PROJ_ORTHOGRAPHIC, 'orthographic'), (L.PROJ_AZIMUTHAL_EQUAL_AREA, 'azimuthal equal area')):
        cc = c if kind == L.PROJ_ORTHOGRAPHIC else np.linspace(-1.01, 1.01, size)
        xx, yy = np.meshgrid(cc, cc)
        xd, yd = L.to_device(xx), L.to_device(yy)
        holder = {}

        def proj():
            holder['ll'] = L.proj_inverse(kind, bc.r_eq, bc.r_polar, 0.0, 30.0, bc.lon_sign, xd, yd)
        proj_ms = timed(proj)
        lon, lat = holder['ll']
        lon = torch.remainder(lon, 360.0)
        mmask = L.mask_from_names(names + ['PIXEL-X', 'PIXEL-Y', 'EMISSION'])
        mout = torch.empty((L.popcount(mmask), size, size), dtype=torch.float64, device='cuda')
        map_ms = timed(lambda: L.backplanes_map(fd[0], lon, lat, mmask, out=mout))
        res[name] = {'size': size, 'proj_inverse_ms': proj_ms, 'backplanes_map_ms': map_ms,
                     'mcells_per_s': size * size / (proj_ms + map_ms) / 1e3,
                     'cells_on_body': int(torch.isfinite(lon).sum())}
    return res


def bench_save_observation(L, torch, pm, bc, sz=2048):
    """SURVEY 8(f) rank 1: Observation.save_observation of a 2048 x 2048 frame, all 26 backplanes
    + the image itself = 27 float64 HDUs (906 MB file).  Reports the three stages separately:
    the fused backplane launch, the big-endian staging launch (HBM-bound: 16 B per element) and
    the single device->host copy of the file image, then the whole call including the disk write."""
    import tempfile
    import time

    from planetmapper_b200 import fits_stage as FS

    img = np.random.default_rng(3).normal(1.0, 0.1, (1, sz, sz))
    obs = pm.Observation(data=img, constants=bc)
    data_dev = obs._get_data_device()
    have, planes = obs.get_backplanes_img_device(L.ALL_PLANES)
    hdus = [FS.ImageHDU(data_dev)] + [FS.ImageHDU(planes[i], name=L.PLANE_NAMES[i]) for i in range(planes.shape[0])]
    headers, hoff, doff, size = FS.file_layout(hdus)
    arrays = [h.data for h in hdus]
    image = torch.empty(size, dtype=torch.uint8, device='cuda')
    host = torch.empty(size, dtype=torch.uint8, pin_memory=True)

    def timed(fn, reps=10):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    stage_ms = timed(lambda: L.fits_stage(arrays, doff, image))
    copy_ms = timed(lambda: host.copy_(image, non_blocking=True), reps=5)
    fd = obs._frame_dev().reshape(1, -1)
    out = torch.empty((1, L.N_PLANES, sz, sz), dtype=torch.float64, device='cuda')
    planes_ms = timed(lambda: L.backplanes_img(fd, sz, sz, L.ALL_PLANES, out=out))
    n_elems = sum(a.numel() for a in arrays)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, 'nav.fits')
        obs.save_observation(path, print_info=False)   # warm (page cache, pinned allocator)
        obs._clear_cache()
        t0 = time.perf_counter()
        obs.save_observation(path, print_info=False)
        call_s = time.perf_counter() - t0
        file_bytes = os.path.getsize(path)
    return {'workload': f'save_observation: {sz}x{sz} frame, 27 float64 HDUs (image + 26 backplanes)',
            'file_bytes': file_bytes, 'backplanes_26_ms': planes_ms, 'stage_ms': stage_ms,
            'stage_gb_per_s': 16.0 * n_elems / stage_ms / 1e6, 'd2h_ms': copy_ms,
            'd2h_gb_per_s': size / copy_ms / 1e6, 'launches': 2,
            'whole_call_s_incl_disk_write': call_s}


def bench_point_transforms(L, torch, bc, n=10_000_000):
    """SURVEY 8(a) row a18: the vectorised point transforms (xy2lonlat / lonlat2xy over arrays,
    base.py:718-757 in the reference: np.nditer + one ctypes call per element), n points each."""
    fr = c2_frame(bc)
    fd = L.to_device(fr)
    g = torch.Generator(device='cuda').manual_seed(1)
    x = torch.rand(n, dtype=torch.float64, device='cuda', generator=g) * SZ
    y = torch.rand(n, dtype=torch.float64, device='cuda', generator=g) * SZ
    lon = torch.rand(n, dtype=torch.float64, device='cuda', generator=g) * 360.0
    lat = torch.rand(n, dtype=torch.float64, device='cuda', generator=g) * 180.0 - 90.0

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    t_fwd = timed(lambda: L.xy2lonlat(fd, x, y))
    t_inv = timed(lambda: L.lonlat2xy(fd, lon, lat, True))
    t_alt = timed(lambda: L.lonlat2xy(fd, lon, lat, True, alt=1000.0))
    return {'workload': f'{n} random points on the C2 frame', 'xy2lonlat_mpoints_per_s': n / t_fwd / 1e3,
            'lonlat2xy_mpoints_per_s': n / t_inv / 1e3, 'lonlat2xy_alt_raycast_mpoints_per_s': n / t_alt / 1e3}


def bench_time_series(L, torch, pm, rank, world, n_frames=4096, batch=32):
    """C5: the time series of BASELINE.json - 4096 frames of 1024 x 1024, 60 s apart, ending one
    hour before the fixture epoch, sharded by frame across ranks: the 12-plane stack per frame in
    batched launches (one device buffer reused per batch: the full series would be 412 GB of
    planes) plus a 1 deg rectangular nearest reprojection of one synthetic image per frame.
    Europa has no SPK segment in the bundled kernels (SURVEY section 0), so its position comes from the
    analytic orbit about the Jupiter barycentre of planetmapper_b200/minispice/kepler.py (SURVEY 8(d) C5
    option ii) while radii (triaxial: 1562.6 / 1560.3 / 1559.5 km) and the IAU orientation model are the
    PCK's own.  The per-frame host constants are extracted by `planetmapper_b200.series` over host processes
    and reported separately."""
    from planetmapper_b200 import frame as F
    from planetmapper_b200.shard import shard_range

    from planetmapper_b200 import series as S

    sz = 1024
    lo, hi = shard_range(n_frames, rank, world)
    prov = pm.get_default_provider()
    et_end = prov.utc2et('2005-01-01T00:00:00') - 3600.0
    ets = et_end - 60.0 * (n_frames - 1 - np.arange(lo, hi))
    disc = dict(nx=sz, ny=sz, x0=(sz - 1) / 2, y0=(sz - 1) / 2, r0=0.45 * sz, rotation_radians=0.0)
    # host constants: one serial sample for the per-frame cost, then the whole shard over host processes
    t0 = time.perf_counter()
    S.build_series_frames('Europa', ets[:16], 'EARTH', workers=1, kepler=True, **disc)
    serial_ms_per_frame = (time.perf_counter() - t0) / min(16, len(ets)) * 1e3
    S.build_series_frames('Europa', ets[:16 * S.default_workers()], 'EARTH', kepler=True, **disc)   # starts every worker process
    t0 = time.perf_counter()
    frames = S.build_series_frames('Europa', ets, 'EARTH', kepler=True, **disc)
    host_s = time.perf_counter() - t0
    host_workers = S.default_workers()
    S.shutdown_pool()
    fd = L.to_device(frames)
    mask = plane_mask(C2_NAMES)
    out = torch.empty((batch, len(C2_NAMES), sz, sz), dtype=torch.float64, device='cuda')
    lons = np.arange(0.5, 360, 1.0)[::-1]
    lats = np.arange(-89.5, 90, 1.0)
    lo_g, la_g = np.meshgrid(lons, lats)
    # one synthetic image per frame (1 % NaN pixels), resident on the device like the frames
    imgs = torch.empty((hi - lo, sz, sz), dtype=torch.float64, device='cuda')
    for s in range(0, hi - lo, 128):
        part = torch.rand(imgs[s:s + 128].shape, dtype=torch.float64, device='cuda')
        part[torch.rand(part.shape, device='cuda') < 0.01] = float('nan')
        imgs[s:s + 128] = part
    del part
    mapped = torch.empty((hi - lo,) + lo_g.shape, dtype=torch.float64, device='cuda')

    def one_pass():
        for s in range(0, hi - lo, batch):
            n = min(batch, hi - lo - s)
            L.backplanes_img(fd[s:s + n], sz, sz, mask, out=out[:n])

    def reproject():
        S.map_series(frames, imgs, sz, sz, lo_g, la_g, interpolation='linear', batch=batch, out=mapped)
    one_pass()
    reproject()
    torch.cuda.synchronize()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    one_pass()
    e1.record()
    reproject()
    e2.record()
    torch.cuda.synchronize()
    return {'workload': f'C5: {n_frames} Europa / EARTH frames (triaxial; analytic orbit, PCK radii and orientation) of {sz}x{sz}, 60 s apart, 12-plane stack in '
                        f'batches of {batch} frames + map_img(img, degree_interval=1) (linear) of one image per frame, batched '
                        f'(series.map_series); frames {lo}..{hi} on this rank',
            'frames_this_rank': hi - lo, 'host_constants_s': host_s, 'host_workers': host_workers,
            'host_constants_serial_ms_per_frame': serial_ms_per_frame,
            'backplanes_ms': e0.elapsed_time(e1), 'backplanes_mpix_per_s': (hi - lo) * sz * sz / e0.elapsed_time(e1) / 1e3,
            'reprojection_ms': e1.elapsed_time(e2), 'reprojection_frames_per_s': (hi - lo) / e1.elapsed_time(e2) * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--skip-cube', action='store_true', help='skip the mapped-cube (C4) section')
    ap.add_argument('--skip-cpu', action='store_true', help='skip the bounded CPU baselines')
    ap.add_argument('--skip-extra', action='store_true', help='skip the C3 (Saturn rings) and C5 (time series) sections')
    ap.add_argument('--cpu-child', type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_child:
        print(cpu_port_mpix(args.cpu_child, repeats=2)[0])
        return 0
    if args.impl == 'reference':
        return run_reference(args)

    # stdout carries exactly ONE JSON line.  Libraries write to file descriptor 1 behind Python's back
    # (NCCL prints its version banner there at NCCL_DEBUG=VERSION / WARN), so descriptor 1 is pointed at
    # stderr for the whole run and the result goes to a private duplicate of the original stdout.
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    import torch

    import planetmapper_b200 as pm
    from planetmapper_b200 import _lib as L
    from planetmapper_b200.shard import bind_rank_to_cores, env_rank_world, max_over_ranks

    rank, local_rank, world = env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device; there is no CPU fallback')
    torch.cuda.set_device(local_rank)
    # every rank gets its own host cores (and its GPU's NUMA node where the host has more than one) BEFORE it
    # allocates pinned memory
    binding = bind_rank_to_cores(local_rank, int(os.environ.get('LOCAL_WORLD_SIZE', world)), local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    L.load_library()
    bc = load_bc()
    fr = c2_frame(bc)
    mask = plane_mask(C2_NAMES)
    k = len(C2_NAMES)
    out = torch.empty((k, SZ, SZ), dtype=torch.float64, device='cuda')

    # ---- kernel path: the frame constants ride in the launch, planes stay in HBM ----------
    W = max(args.warmup, 3)
    for _ in range(W):
        L.backplanes_img_host(fr, SZ, SZ, mask, out=out)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    launches0 = L.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        L.backplanes_img_host(fr, SZ, SZ, mask, out=out)
    e1.record()
    barrier()
    launches = L.launch_count() - launches0
    ms = e0.elapsed_time(e1) / args.steps
    ms = max_over_ranks(ms, world, device='cuda')
    value = world * SZ * SZ / (ms * 1e-3) / 1e6

    # ---- end to end through the public API, host arrays out ---------------------------------
    e2e_steps = max(3, min(args.steps, 10))
    nbytes = k * SZ * SZ * 8

    def e2e_dropin():
        # the reference's own call sequence (body_xy.py:2586-2630): one get_backplane_img per name
        body = pm.BodyXY(constants=bc, nx=SZ, ny=SZ)      # fresh object: empty caches
        planes = {n: body.get_backplane_img(n) for n in C2_NAMES}
        return float(planes['EMISSION'][SZ // 2, SZ // 2])

    pinned = torch.empty((k, SZ, SZ), dtype=torch.float64).pin_memory()

    def e2e_batched():
        body = pm.BodyXY(constants=bc, nx=SZ, ny=SZ)
        planes = body.get_backplane_imgs(C2_NAMES, out=pinned)
        return float(planes['EMISSION'][SZ // 2, SZ // 2])

    def timed_host(fn, steps):
        import gc

        for _ in range(2):
            fn()
        barrier()
        gc.collect()
        gc.freeze()       # torch's import graph leaves the collector's view: no 50 ms generation-2 pass mid-loop
        try:
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
            t = (time.perf_counter() - t0) / steps * 1e3
        finally:
            gc.unfreeze()
        return max_over_ranks(t, world, device='cuda')

    e2e_ms = timed_host(e2e_dropin, e2e_steps)
    e2e_batched_ms = timed_host(e2e_batched, e2e_steps)

    # the ceiling of any end-to-end number: the same bytes, device -> pinned host, all ranks at once
    def raw_copy():
        pinned.copy_(out, non_blocking=True)
    for _ in range(2):
        raw_copy()
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(5):
        raw_copy()
    c1.record()
    torch.cuda.synchronize()
    d2h_ms = max_over_ranks(c0.elapsed_time(c1) / 5, world, device='cuda')
    clocks = sampler.stop() if rank == 0 else None
    e2e_value = world * SZ * SZ / (e2e_ms * 1e-3) / 1e6

    result = None
    if rank == 0:
        planes_host = out[0].cpu().numpy()
        # plane 0 of the packed output is LON-GRAPHIC (lowest id); its NaN mask = on-disc mask
        flops, classes = algorithmic_flops_per_frame(planes_host, fr)
        fp64_peak = L.fp64_peak_probe()
        fp64_peak_3reg = L.fp64_peak_probe(kind=1)
        achieved = flops / (ms * 1e-3) / 1e12
        result = {
            'metric': METRIC, 'value': value, 'unit': 'Mpix/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': W, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': WORKLOAD,
                       'l2': 'each step writes 403 MB of planes (> 126 MB L2); no flush needed',
                       'frames_per_step_per_gpu': 1, 'parallelism': f'frames sharded, {world} rank(s), no collective',
                       'launch': 'pm_backplanes_img_host: the 92 frame constants + derived values are a kernel '
                                 'parameter (constant bank); no host -> device copy is enqueued',
                       'host_binding': binding},
            'gpu_launches': int(launches),
            'e2e': {'value': e2e_value, 'unit': 'Mpix/s', 'ms_per_step': e2e_ms,
                    'h2d_bytes_per_step': int(fr.nbytes), 'd2h_bytes_per_step': int(nbytes),
                    'api': 'drop-in: BodyXY(constants=...) then get_backplane_img(name) for each of the 12 names '
                           '(1 kernel launch, 12 device -> pinned-host copies - the last 10 read ahead on a side '
                           'stream - 12 owned float64 arrays returned); gc.freeze() before timing',
                    'steps': e2e_steps,
                    'batched': {'value': world * SZ * SZ / (e2e_batched_ms * 1e-3) / 1e6, 'ms_per_step': e2e_batched_ms,
                                'api': 'BodyXY.get_backplane_imgs(12 names, out=pinned): 1 launch, 1 copy'},
                    'd2h_ceiling': {'ms_per_step': d2h_ms, 'gb_per_s_per_gpu': nbytes / (d2h_ms * 1e-3) / 1e9,
                                    'gb_per_s_all_gpus': world * nbytes / (d2h_ms * 1e-3) / 1e9,
                                    'value': world * SZ * SZ / (d2h_ms * 1e-3) / 1e6,
                                    'what': 'cudaMemcpyAsync of the same 403 MB, device -> pinned host, all ranks '
                                            'concurrently, max over ranks: no end-to-end number can exceed it'},
                    'frac_of_d2h_ceiling': d2h_ms / e2e_ms},
            'roofline': {'bound': 'fp64', 'achieved': achieved, 'peak': fp64_peak, 'unit': 'TFLOP/s',
                         'frac': achieved / fp64_peak, 'traffic': ncu_traffic('backplanes_img_c2'),
                         'peak_source': 'pm_fp64_probe(kind 0): 8 independent DFMA chains/thread with ONE register '
                                        'operand each, full grid, measured in this run (MEASURED_PEAKS.json has no '
                                        'FP64 entry)',
                         'operand_limited': {
                             'peak_3_register_dfma': fp64_peak_3reg, 'frac': achieved / fp64_peak_3reg,
                             'what': 'pm_fp64_probe(kind 1): the same probe with three DISTINCT register operands '
                                     'per DFMA, the form dot / cross / axpy of per-pixel vectors issue.  The '
                                     'register file needs 3 cycles to deliver their six 32-bit sources, the pipe '
                                     'issues a DFMA every 2: such code tops out at 2/3 of `peak` '
                                     '(tools/microbench/fp64_operands.cu, profiles/r2_summary.md)'},
                         'issue_model': issue_model(classes, ms, clocks, torch.cuda.get_device_properties(0).multi_processor_count),
                         'algorithmic_flops_per_launch': flops, 'pixel_classes': classes,
                         'hbm_bytes_per_launch_algorithmic': int(nbytes),
                         # the same launch seen as an HBM kernel (why the bound is the FP64 pipe, not memory)
                         'hbm_view': {'bound': 'hbm', 'achieved': nbytes / (ms * 1e-3) / 1e9,
                                      'peak': measured_peaks()[0]['hbm_gbs'], 'unit': 'GB/s',
                                      'frac': nbytes / (ms * 1e-3) / 1e9 / measured_peaks()[0]['hbm_gbs']},
                         'note': 'frac counts executed flops (FMA = 2, MUL / ADD = 1) against the one-register-operand '
                                 'DFMA peak; see operand_limited for what the pipe sustains on three-register DFMAs.  The kernel '
                                 'is ISSUE bound: an FP64 instruction holds the issue port 2 (3) cycles and the non-FP64 '
                                 'instructions (45 % of the stream: selects, constant loads, moves, addresses) are not hidden '
                                 'behind it (tools/microbench/fp64_operands.cu, DESIGN.md 3.4): 138 - 160 M of the 168 M '
                                 'sub-partition cycles of a launch are issue cycles',
                         'ncu': ncu_summary('backplanes_img_c2')},
            'clocks': clocks,
        }
    if not args.skip_cube:
        cube_res = bench_mapped_cube(L, torch, pm, bc, rank, world)
        if rank == 0:
            result['mapped_cube'] = cube_res
    if not args.skip_extra:
        ts = bench_time_series(L, torch, pm, rank, world)
        t_all = max_over_ranks(ts['backplanes_ms'], world, device='cuda')
        t_map = max_over_ranks(ts['reprojection_ms'], world, device='cuda')
        if rank == 0:
            ts['backplanes_mpix_per_s_all_ranks'] = 4096 * 1024 * 1024 / t_all / 1e3
            ts['reprojection_frames_per_s_all_ranks'] = 4096 / t_map * 1e3
            ts['scaling'] = 'strong'
            result['time_series'] = ts
            result['saturn_rings'] = bench_saturn_rings(L, torch, pm)
            result['save_observation'] = bench_save_observation(L, torch, pm, bc)
            result['point_transforms'] = bench_point_transforms(L, torch, bc)
    if rank == 0:
        if not args.skip_cpu and world == 1:  # the CPU baselines are N = 1 measurements
            mp, dt = cpu_port_mpix(CPU_SAMPLE_SZ, repeats=3)
            one = cpu_one_core_mpix()
            result['cpu_baseline'] = {
                'value': mp, 'unit': 'Mpix/s', 'cores': omp_threads(), 'kind': 'port',
                'sample': f'the full C2 frame ({CPU_SAMPLE_SZ}x{CPU_SAMPLE_SZ}, 12 planes), best of 3 passes '
                          f'({dt:.2f} s wall each on {omp_threads()} OpenMP threads)',
                'one_core': {'value': one, 'unit': 'Mpix/s', 'cores': 1,
                             'sample': 'the C2 geometry at 1024 x 1024 (same disc fraction), OMP_NUM_THREADS=1'},
                'note': 'C restatement in oracle/ (the Python+spiceypy reference is not installable here; '
                        'it is ~3 orders of magnitude slower than this port, SURVEY.md section 6)'}
            if not args.skip_extra:
                result['cpu_baseline']['other_configs'] = cpu_baselines_extra(bc)
        os.write(result_fd, (json.dumps(result) + '\n').encode())
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
