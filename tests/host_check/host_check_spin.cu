// host_check_spin.cu - TEST INFRASTRUCTURE ONLY.
//
// Host instantiation of both paths of pm::image_point (planetmapper_b200/csrc/pm_device.cuh): the
// general one, which spins the observer, the ray and the Sun to every epoch, and the one the launchers
// pick for frames with FrameD::spin_sym, which works in the body frame at t_ref.  Lets the non-GPU
// suite compare the two on the same frame whatever its flag says.  Built by tests/test_spin_sym_host.py
// into a temporary directory; never linked into or loaded by libpm_b200.so.
#include <cstdint>

#include "../../planetmapper_b200/csrc/pm_device.cuh"

namespace {
struct ArraySink {
    double *v;
    void put(int k, double val) { v[k] = val; }
};
}  // namespace

extern "C" {

// FrameD::spin_sym of the frame, as load_frame_host derives it
int hc_spin_sym(const PMFrame *frame) {
    pm::FrameD fs;
    pm::load_frame_host(fs, frame);
    return fs.spin_sym;
}

// out: [26][n] (all plane ids, unrequested planes NaN); spin_sym selects the path, not the frame's flag
int hc_backplanes_points_path(const PMFrame *frame, const double *x, const double *y, int64_t n, uint64_t mask,
                              int spin_sym, double *out) {
    pm::FrameD fs;
    pm::load_frame_host(fs, frame);
    for (int64_t i = 0; i < n; i++) {
        double v[PM_N_PLANES];
        for (int k = 0; k < PM_N_PLANES; k++) v[k] = NAN;
        ArraySink sink{v};
        if (spin_sym)
            pm::image_point<true, false, true>(fs, x[i], y[i], mask, sink);
        else
            pm::image_point<true, false, false>(fs, x[i], y[i], mask, sink);
        for (int k = 0; k < PM_N_PLANES; k++) out[k * n + i] = v[k];
    }
    return 0;
}
}
