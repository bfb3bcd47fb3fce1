"""
The frame kinds of the single-frame image kernel and the local-solar-time table, on the CPU
(tests/host_check/host_check_kind.cu):

- frame_kind picks kFrameSpinZ (spin_z and biaxial fixed at compile time) for Jupiter, Saturn and Venus,
  kFrameSpinSym for a sphere with a tilted spin axis and kFrameGeneral for triaxial bodies; and image_pixel
  instantiated for kFrameSpinZ gives the same bits as the kFrameSpinSym instantiation, which tests those
  flags at run time (the batched kernel's path);
- the local-solar-time fractions mn / 60 and sc / 3600 read from a table equal the correctly rounded
  quotients, which the division they replace produced, for all 3600 (mn, sc) pairs.
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import img_case, triaxial_constants
from planetmapper_b200 import frame as F
from test_spin_sym_host import _bc

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'host_check', 'host_check_kind.cu')
GENERAL, SPIN_SYM, SPIN_Z = 0, 1, 2


@pytest.fixture(scope='module')
def kind_lib(tmp_path_factory):
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not available')
    so = str(tmp_path_factory.mktemp('host_check_kind') / 'libpm_hostcheck_kind.so')
    subprocess.run([nvcc, '-O2', '-std=c++17', '-shared', '-Xcompiler', '-fPIC', '-Wno-deprecated-gpu-targets',
                    '-o', so, SRC], check=True, capture_output=True)
    lib = ctypes.CDLL(so)
    lib.hc_local_solar_time.restype = ctypes.c_double
    lib.hc_local_solar_time.argtypes = [ctypes.c_void_p, ctypes.c_double]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def flags(lib, fr):
    out = np.zeros(4, dtype=np.int32)
    assert lib.hc_frame_flags(_p(np.ascontiguousarray(fr, dtype=np.float64)), _p(out)) == 0
    return dict(zip(('spin_sym', 'spin_z', 'biaxial', 'kind'), out.tolist()))


def _frame(bc):
    return img_case(bc, 64, 48, 31.0, 24.5, 20.0, 17.0)


def test_frame_kinds(kind_lib, bc_hst):
    for bc in (bc_hst, _bc('Saturn', 'EARTH'), _bc('Venus', 'EARTH')):
        f = flags(kind_lib, _frame(bc))
        assert f['kind'] == SPIN_Z and f['spin_z'] and f['biaxial'], f
    for kind in ('europa', 'triaxial-x'):
        assert flags(kind_lib, _frame(triaxial_constants(kind)))['kind'] == GENERAL, kind
    tilted = _frame(_bc('Venus', 'EARTH'))
    w = F.frame_field(tilted, 'omega')
    w[:] = np.linalg.norm(w) * np.array([np.sin(0.3), 0.0, np.cos(0.3)])
    f = flags(kind_lib, tilted)
    assert f['kind'] == SPIN_SYM and not f['spin_z'], f


def _stack(lib, fr, x, y, kind):
    out = np.empty((26, x.size))
    assert lib.hc_stack_kind(_p(np.ascontiguousarray(fr)), _p(x), _p(y), ctypes.c_int64(x.size), ctypes.c_int(kind),
                             _p(out)) == 0
    return out


def test_spin_z_kind_equals_runtime_kind(kind_lib, bc_hst):
    sz = 2048
    c = (sz - 1) / 2
    fr = img_case(bc_hst, sz, sz, c, c, 0.9 * c, 0.0)
    assert flags(kind_lib, fr)['kind'] == SPIN_Z
    rng = np.random.default_rng(6)
    x, y = rng.integers(0, sz, 20000).astype(float), rng.integers(0, sz, 20000).astype(float)
    # limb pixels, where sincpt iterates to convergence
    t = rng.uniform(0.0, 2.0 * np.pi, 4000)
    x = np.concatenate([x, np.round(c + 0.9 * c * np.cos(t))])
    y = np.concatenate([y, np.round(c + 0.9 * c * np.sin(t))])
    a, b = _stack(kind_lib, fr, x, y, SPIN_Z), _stack(kind_lib, fr, x, y, SPIN_SYM)
    assert np.isfinite(a[0]).sum() > 10000
    assert np.array_equal(a.view(np.int64), b.view(np.int64))


def test_lst_fractions_are_correctly_rounded(kind_lib):
    got = np.empty(2)
    mn, sc = np.meshgrid(np.arange(60), np.arange(60), indexing='ij')
    qm, qs = np.empty(mn.shape), np.empty(mn.shape)
    for i in range(60):
        for j in range(60):
            kind_lib.hc_lst_fractions(ctypes.c_int(i), ctypes.c_int(j), _p(got))
            qm[i, j], qs[i, j] = got
    assert np.array_equal(qm, mn / 60.0) and np.array_equal(qs, sc / 3600.0)


def test_local_solar_time_whole_seconds(kind_lib, bc_hst):
    """every whole second of a local day: hr + mn / 60 + sc / 3600 with the reference's two roundings"""
    fr = np.ascontiguousarray(_frame(bc_hst))
    lon_sign = float(F.frame_field(fr, 'lon_sign')[0])
    prograde = float(F.frame_field(fr, 'prograde')[0])
    sun = float(F.frame_field(fr, 'sun_lon_lst')[0])
    secs = np.arange(0, 86400, 7) + 0.5   # mid-second: away from the floor's rounding edge
    ang = (secs - 43200.0) / 86400.0 * 2.0 * np.pi
    ang = ang if prograde != 0.0 else -ang
    lon = np.rad2deg((ang + sun) * lon_sign)
    got = np.array([kind_lib.hc_local_solar_time(_p(fr), float(v)) for v in lon])
    isec = np.floor(secs).astype(np.int64)
    hr, rem = np.divmod(isec, 3600)
    mn, sc = np.divmod(rem, 60)
    want = (hr + mn / 60.0) + sc / 3600.0
    assert np.array_equal(got, want)
