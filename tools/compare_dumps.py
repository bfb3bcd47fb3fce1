#!/usr/bin/env python
"""Compares two `bench.py --dump-outputs DIR` directories (C2 planes at the same sampled pixels) plane by
plane, in the layout of profiles/r*_dump_compare.txt:   python tools/compare_dumps.py PARENT_DIR NEW_DIR"""
import os
import sys

import numpy as np


def main(a_dir, b_dir):
    on_a = np.load(os.path.join(a_dir, 'ON-DISC.npy')) > 0
    on_b = np.load(os.path.join(b_dir, 'ON-DISC.npy')) > 0
    print('ON-DISC identical:', bool(np.array_equal(on_a, on_b)), 'n on-disc', int(on_a.sum()), int(on_b.sum()))
    on = on_a & on_b
    em = np.load(os.path.join(a_dir, 'EMISSION.npy'))[on]
    inc = np.load(os.path.join(a_dir, 'INCIDENCE.npy'))[on]
    for f in sorted(os.listdir(a_dir)):
        name = f[:-4]
        if name == 'ON-DISC':
            continue
        a, b = np.load(os.path.join(a_dir, f))[on], np.load(os.path.join(b_dir, f))[on]
        d = np.abs(a - b)
        if name.startswith('LON'):   # 0 and 360 deg are the same longitude
            d = np.minimum(d, 360.0 - d)
        i = int(np.argmax(d))
        rel = d / np.maximum(np.abs(a), np.finfo(float).tiny)
        low = em < 80.0
        print(f'{name:<17s} max_abs {d[i]:.3e} max_rel {rel.max():.3e} | at emission {em[i]:.3f} incidence {inc[i]:.3f}'
              f' | emission<80: max_abs {d[low].max():.3e} | bit-identical {int((a == b).sum())} / {a.size}')


if __name__ == '__main__':
    main(*sys.argv[1:3])
