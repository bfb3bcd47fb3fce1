// host_check_regrid.cu - TEST INFRASTRUCTURE ONLY.
//
// Host instantiation of the smoothing-spline fit of pm_regrid_fit (planetmapper_b200/csrc/pm_regrid.cuh):
// the same fpregr / fpgrre code the device runs, with a serial executor, so the non-GPU suite can hold
// the knot logic against scipy's FITPACK (including runs with capped nxest / nyest) and the GPU suite
// can hold the device fit against it bit for bit.  Built by the tests into a temporary directory; never
// linked into or loaded by libpm_b200.so.
#include <cstdint>
#include <vector>

#include "../../planetmapper_b200/csrc/pm_regrid.cuh"

namespace {
struct SerialExec {
    template <class F>
    PMR_HD void each(int n, F f) const {
        for (int j = 0; j < n; j++) f(j);
    }
    template <class F>
    PMR_HD void one(F f) const {
        f();
    }
    template <class F>
    PMR_HD void lane(int, F f) const {
        f();
    }
    PMR_HD void sync() const {}
};
struct RowMajor {
    const double *z;
    int my;
    PMR_HD double operator()(int i, int j) const { return z[(int64_t)i * my + j]; }
};
}  // namespace

extern "C" {

// z: [mx][my] row-major (RectBivariateSpline's z with x = arange(mx), y = arange(my)).
// tx[nxest], ty[nyest], c[(nxest-kx-1)(nyest-ky-1)]; out_n = {nx, ny, ier}; *fp.
int hc_regrid_fit(const double *z, int mx, int my, int kx, int ky, double s, int nxest, int nyest, int maxit,
                  double *tx, double *ty, double *c, int *out_n, double *fp) {
    using namespace pm::regrid;
    const int nxe = nxest > 2 * (kx + 1) ? nxest : 2 * (kx + 1), nye = nyest > 2 * (ky + 1) ? nyest : 2 * (ky + 1);
    std::vector<double> d((size_t)work_doubles(mx, my, kx, ky, nxe, nye));
    std::vector<int> iw((size_t)work_ints(mx, my, nxe, nye));
    Work w = carve(d.data(), iw.data(), mx, my, kx, ky, nxe, nye);
    Ctl ctl;
    double rot[3 * (kMaxK + 2)];
    double fp_slot = 0.0;
    fit_plane(SerialExec{}, RowMajor{z, my}, mx, my, kx, ky, s, nxest, nyest, maxit, tx, ty, c, w, ctl, rot, &fp_slot,
              out_n, fp);
    return 0;
}

// bispeu of one fitted plane at n points (x along the slow axis).
int hc_regrid_eval(const double *tx, int nx, const double *ty, int ny, const double *c, int kx, int ky,
                   const double *x, const double *y, int64_t n, double *out) {
    for (int64_t i = 0; i < n; i++) out[i] = pm::regrid::evaluate(tx, nx, ty, ny, c, kx, ky, x[i], y[i]);
    return 0;
}
}
