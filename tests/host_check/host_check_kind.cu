// host_check_kind.cu - TEST INFRASTRUCTURE ONLY.
//
// Host instantiation of the pieces of planetmapper_b200/csrc/pm_device.cuh that pick and serve the image
// kernel's frame kinds: the flags and kind of a frame, the local-solar-time fraction table and image_pixel
// for each kind.  Built by tests/test_frame_kind_host.py into a temporary directory; never linked into or
// loaded by libpm_b200.so.
#include <cstdint>

#include "../../planetmapper_b200/csrc/pm_device.cuh"

namespace {
struct ArraySink {
    double *v;
    void put(int k, double val) { v[k] = val; }
};
constexpr uint64_t kStack = pm::kLonLatMask | pm::kCentricMask | pm::kIllumMask | pm::kStateMask;
}  // namespace

extern "C" {

// flags[0..3]: spin_sym, spin_z, biaxial, frame_kind
int hc_frame_flags(const PMFrame *frame, int *flags) {
    pm::FrameD fs;
    pm::load_frame_host(fs, frame);
    flags[0] = fs.spin_sym;
    flags[1] = fs.spin_z;
    flags[2] = fs.biaxial;
    flags[3] = pm::frame_kind(fs);
    return 0;
}

// out[0] = mn / 60, out[1] = sc / 3600 as local_solar_time reads them
void hc_lst_fractions(int mn, int sc, double *out) { pm::lst_fractions(mn, sc, out[0], out[1]); }

// local_solar_time of a planetographic longitude in degrees
double hc_local_solar_time(const PMFrame *frame, double lon_deg) { return pm::local_solar_time(*frame, lon_deg); }

// out: [26][n] of the default 12-plane stack, image_pixel instantiated for kind (the single-frame image
// kernel's per-pixel code), whatever the frame's own kind
int hc_stack_kind(const PMFrame *frame, const double *x, const double *y, int64_t n, int kind, double *out) {
    pm::FrameD fs;
    pm::load_frame_host(fs, frame);
    for (int64_t i = 0; i < n; i++) {
        double v[PM_N_PLANES];
        for (int k = 0; k < PM_N_PLANES; k++) v[k] = NAN;
        ArraySink sink{v};
        if (kind == pm::kFrameSpinZ)
            pm::image_pixel<false, kStack, false, pm::kFrameSpinZ>(fs, x[i], y[i], kStack, sink);
        else if (kind == pm::kFrameSpinSym)
            pm::image_pixel<false, kStack, false, pm::kFrameSpinSym>(fs, x[i], y[i], kStack, sink);
        else
            pm::image_pixel<false, kStack, false, pm::kFrameGeneral>(fs, x[i], y[i], kStack, sink);
        for (int k = 0; k < PM_N_PLANES; k++) out[k * n + i] = v[k];
    }
    return 0;
}
}
