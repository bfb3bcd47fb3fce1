// host_check_spinz.cu - TEST INFRASTRUCTURE ONLY.
//
// FrameD::spin_z as load_frame_host derives it, for tests/test_atan_table.py.  Built by that test into a
// temporary directory; never linked into or loaded by libpm_b200.so.
#include "../../planetmapper_b200/csrc/pm_device.cuh"

extern "C" int hc_spin_z(const PMFrame *frame) {
    pm::FrameD fs;
    pm::load_frame_host(fs, frame);
    return fs.spin_z;
}
