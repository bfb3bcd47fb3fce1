// host_check_points.cu - TEST INFRASTRUCTURE ONLY.
//
// Host instantiation of pm::image_point, the per-point code of pm_backplanes_points_host
// (planetmapper_b200/csrc/pm_device.cuh), so the non-GPU suite can run it on the CPU: the guard
// that keeps non-finite positions away from sincpt, and the ring-plane switch of
// PM_FLAG_RING_ALL.  Built by tests/test_points_host.py into a temporary directory; never
// linked into or loaded by libpm_b200.so.
#include <cstdint>

#include "../../planetmapper_b200/csrc/pm_device.cuh"

namespace {
struct ArraySink {
    double *v;
    void put(int k, double val) { v[k] = val; }
};
}  // namespace

extern "C" {

// out: [26][n] (all plane ids, unrequested planes NaN); flags as pm_backplanes_points_host
int hc_backplanes_points(const PMFrame *frame, const double *x, const double *y, int64_t n, uint64_t mask,
                         uint32_t flags, double *out) {
    pm::FrameD fs;
    pm::load_frame_host(fs, frame);
    for (int64_t i = 0; i < n; i++) {
        double v[PM_N_PLANES];
        for (int k = 0; k < PM_N_PLANES; k++) v[k] = NAN;
        ArraySink sink{v};
        if (!(mask & pm::kSkyMask))
            pm::image_point<false, false>(fs, x[i], y[i], mask, sink);
        else if (flags & PM_FLAG_RING_ALL)
            pm::image_point<true, true>(fs, x[i], y[i], mask, sink);
        else
            pm::image_point<true, false>(fs, x[i], y[i], mask, sink);
        for (int k = 0; k < PM_N_PLANES; k++) out[k * n + i] = v[k];
    }
    return 0;
}
}
