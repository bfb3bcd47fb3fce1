"""MiniSpice (host-side, once-per-frame ephemeris stand-in) against the reference's
known answers, and the bundled extract against itself."""
import math
import os

import numpy as np
import pytest

import planetmapper_b200 as pm
from planetmapper_b200 import frame as F
from planetmapper_b200.minispice import MiniSpice, utc2et
from planetmapper_b200.minispice.textkernel import parse_text_kernel


def test_utc2et_known_answer():
    # tests/test_body.py:110
    assert utc2et('2005-01-01T00:00:00') == pytest.approx(157809664.1839331, abs=1e-7)
    assert utc2et('2000-01-01T12:00:00') == pytest.approx(64.18392728473108, abs=1e-6)
    assert utc2et('2005-01-01') == utc2et('2005-01-01T00:00:00')


def test_subpoint_lon_known_answer_from_extract():
    # tests/test_body.py:39-42: Body('Jupiter', utc='2005-01-01').subpoint_lon
    ms = pm.get_default_provider()
    bc = F.build_body_constants(ms, 'Jupiter', '2005-01-01', 'EARTH')
    assert bc.subpoint_lon == pytest.approx(153.12547767272153, abs=1e-9)
    assert bc.positive_longitude_direction == 'W'
    assert bc.target_id == 599


def test_orientation_is_a_rotation_and_omega_matches_finite_difference():
    ms = pm.get_default_provider()
    if not isinstance(ms, MiniSpice):
        pytest.skip('default provider is spiceypy')
    et = 157806930.0
    r, w = ms.orientation(599, et)
    assert np.allclose(r @ r.T, np.eye(3), atol=1e-14)
    h = 1.0  # truncation ~ omega^3 h^2 / 6 = 9e-13; W (1.6e6 deg) quantisation ~ 2e-12
    rp, _ = ms.orientation(599, et + h)
    rm, _ = ms.orientation(599, et - h)
    drdt = (rp - rm) / (2 * h)
    om = -drdt @ r.T
    w_fd = np.array([om[2, 1], om[0, 2], om[1, 0]])
    assert np.allclose(w, w_fd, rtol=0, atol=1e-11)
    # Jupiter System III: 870.536 deg/day
    assert math.degrees(w[2]) * 86400 == pytest.approx(870.536, abs=1e-6)


def test_text_kernel_parser():
    pool = parse_text_kernel("""
    junk BODY1_X = 5
    \\begindata
      BODY599_RADII = ( 71492   71492   66854 )
      BODY599_PM    = ( 284.95  870.5360000  0. )
      DELTET/K      = 1.657D-3
      NAME          = 'it''s'
      LIST         += ( 1 2 )
      LIST         += 3
    \\begintext
      BODY599_RADII = ( 1 1 1 )
    """)
    assert pool['BODY599_RADII'] == [71492.0, 71492.0, 66854.0]
    assert pool['DELTET/K'] == [1.657e-3]
    assert pool['NAME'] == ["it's"]
    assert pool['LIST'] == [1.0, 2.0, 3.0]
    assert 'BODY1_X' not in pool


def test_saturn_frame_builds_before_spk_edge():
    ms = pm.get_default_provider()
    bc = F.build_body_constants(ms, 'Saturn', '2004-12-30T00:00:00', 'EARTH')
    assert bc.radii[0] == 60268.0 and bc.prograde
    assert 1.1e9 < bc.target_distance < 1.7e9


def test_native_primitives_match_the_python_reader():
    """NativeSpice (pm_host_ssb_state / pm_host_orientation in libpm_b200.so) evaluates the same
    tables with the same formulas: agreement to the last bit or two, same errors, and frames whose
    constants differ only where the formulas themselves amplify rounding (the finite-difference
    acceleration, the ring-plane constant)."""
    from planetmapper_b200.minispice.native import NativeSpice

    py = MiniSpice.from_extract(os.path.join(pm._DATA_DIR, 'ephem_extract.npz'),
                                os.path.join(pm._DATA_DIR, 'pck_pool.json'))
    nat = NativeSpice.from_minispice(py)
    assert isinstance(pm.get_default_provider(), (NativeSpice,)) or not isinstance(pm.get_default_provider(), MiniSpice)
    et0 = utc2et('2005-01-01T00:00:00')
    for body in (10, 399, 301, 599, 699, 499, 299, 199, 5, 3):
        for dt in (-10.0, -1234.5, -86400 * 3.3, -86400 * 5.9):   # the extract ends at 2005-01-01 for some bodies
            a, b = py.ssb_state(body, et0 + dt), nat.ssb_state(body, et0 + dt)
            assert np.allclose(a, b, rtol=2e-14, atol=0), (body, dt, a, b)
    for body in (599, 399, 301, 299, 499, 199, 699):
        for dt in (0.0, -1234.5, -86400 * 3.3):
            (ra, wa), (rb, wb) = py.orientation(body, et0 + dt), nat.orientation(body, et0 + dt)
            assert np.max(np.abs(ra - rb)) < 1e-15 and np.allclose(wa, wb, rtol=1e-13, atol=1e-12 * np.max(np.abs(wa))), (body, dt)
    for bad_call in (lambda p: p.ssb_state(599, et0 + 400 * 86400), lambda p: p.ssb_state(12345, et0)):
        with pytest.raises(LookupError):
            bad_call(py)
        with pytest.raises(LookupError):
            bad_call(nat)
    loose = {'AT': 1e-8, 'ring_c': 1e-9, 'ring_n': 1e-10, 'ang2km': 1e-9, 'km2ang': 1e-9}
    for target, observer in (('Jupiter', 'EARTH'), ('Saturn', 'EARTH'), ('Moon', 'EARTH'), ('Earth', 'MOON')):
        fa = F.pack_frame(F.build_body_constants(py, target, None, observer, et=et0 - 2 * 86400), nx=64, ny=64,
                          x0=31.5, y0=31.5, r0=28.0, rotation_radians=0.3)
        fb = F.pack_frame(F.build_body_constants(nat, target, None, observer, et=et0 - 2 * 86400), nx=64, ny=64,
                          x0=31.5, y0=31.5, r0=28.0, rotation_radians=0.3)
        for name, (o, n) in F.PMFRAME_OFFSETS.items():
            a, b = fa[o:o + n], fb[o:o + n]
            scale = np.max(np.abs(a)) or 1.0
            assert np.max(np.abs(a - b)) / scale <= loose.get(name, 1e-11), (target, name)
