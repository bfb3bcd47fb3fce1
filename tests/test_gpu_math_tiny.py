"""ulp error of the tiny-angle sin / cos tier that the image kernels use for pixel offsets
(pm_math.cuh sincos_tiny, reached through sincos_small2 for |x| <= 2^-8), measured on the
device through pm_math_probe kinds 12 / 13 against numpy long double - the same bars as
the pi/4 polynomial of tests/test_gpu_math.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_device_tiny_sincos_ulp_error():
    import torch

    from planetmapper_b200 import _lib as L

    rng = np.random.default_rng(1)
    n = 1 << 20
    th = rng.uniform(-1.0, 1.0, n) * 2.0 ** rng.uniform(-40, -8, n)
    th[:4] = [2.0 ** -8, -2.0 ** -8, 0.0, 3.0e-4]  # the tier's edge, zero, an arcminute-class offset

    def run(kind):
        out = L.math_probe(kind, L.to_device(th))
        torch.cuda.synchronize()
        return out.cpu().numpy()

    tl = th.astype(np.longdouble)
    s, c = run(12), run(13)
    ws, wc = np.sin(tl), np.cos(tl)
    nz = th != 0.0
    err_s = float(np.max(np.abs(s[nz].astype(np.longdouble) - ws[nz]) / np.spacing(np.abs(th[nz]))))
    err_c = float(np.max(np.abs(c.astype(np.longdouble) - wc) / np.spacing(np.abs(wc.astype(np.float64)))))
    print('tiny sincos ulp errors: sin %.3f cos %.3f' % (err_s, err_c))
    assert err_s <= 1.5 and err_c <= 2.0
    assert s[2] == 0.0 and c[2] == 1.0
