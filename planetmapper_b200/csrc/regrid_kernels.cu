// regrid_kernels.cu - map_img with spline_smoothing > 0: FITPACK's smoothing spline on the image grid
// (RectBivariateSpline(arange(ny), arange(nx), plane, kx, ky, s), body_xy.py:1651-1702), fitted per
// plane on the device, then evaluated at the map cells (bispeu).
//
//   regrid_fit_kernel      one CTA per plane: pm_regrid.cuh's fpregr / fpgrre with the threads of the CTA
//                          on the right-hand-side columns; all-NaN planes are not fitted (nx = ny = 0).
//   gather_regrid_kernel   one (cell, plane) per thread: fpbisp on that plane's own knots, with the NaN
//                          rule of pm_gather (_should_propagate_nan_to_map).
//
// The data are the repaired planes of pm_spline_prepare(degree 1) (plane-quad layout) and its NaN bit
// planes, so the NaN repair is the one every other spline mode uses.
#include "pm_kernels.h"
#include "pm_regrid.cuh"

namespace pm {
namespace {

constexpr int kFitBlock = 128;   // >= 96: lane(0..2) run on three different warps
constexpr int kEvalBlock = 256;

struct BlockExec {
    template <class F>
    PMR_HD void each(int n, F f) const {
#if defined(__CUDA_ARCH__)
        for (int j = threadIdx.x; j < n; j += blockDim.x) f(j);
#endif
    }
    template <class F>
    PMR_HD void one(F f) const {
#if defined(__CUDA_ARCH__)
        if (threadIdx.x == 0) f();
#endif
    }
    template <class F>
    PMR_HD void lane(int k, F f) const {
#if defined(__CUDA_ARCH__)
        if (threadIdx.x == 32 * k) f();
#endif
    }
    PMR_HD void sync() const {
#if defined(__CUDA_ARCH__)
        __syncthreads();
#endif
    }
};

// plane l of the repaired cube in pm_spline_prepare's plane-quad layout; (i, j) = (row, column)
struct QuadPlane {
    const double *base;  // coefq + (l / 4) * ny * nx * 4 + l % 4
    int nx;
    PMR_HD double operator()(int i, int j) const { return base[((int64_t)i * nx + j) * 4]; }
};

struct RegridSlots {
    int nxest, nyest;
    int64_t ncmax, wd, wi;  // coefficients per plane, workspace doubles / ints per plane
};
inline RegridSlots regrid_slots(int ny, int nx, int k_rows, int k_cols) {
    RegridSlots s;
    s.nxest = ny + k_rows + 1;
    s.nyest = nx + k_cols + 1;
    s.ncmax = (int64_t)ny * nx;
    s.wd = regrid::work_doubles(ny, nx, k_rows, k_cols, s.nxest, s.nyest);
    s.wi = regrid::work_ints(ny, nx, s.nxest, s.nyest);
    return s;
}

__global__ void __launch_bounds__(kFitBlock)
    regrid_fit_kernel(const double *__restrict__ coefq, const uint32_t *__restrict__ plane_bits, int ny, int nx,
                      int k_rows, int k_cols, double s, int maxit, RegridSlots sl, double *__restrict__ tx,
                      double *__restrict__ ty, double *__restrict__ c, int *__restrict__ nxy, double *__restrict__ fp,
                      int *__restrict__ ier, double *__restrict__ wd, int *__restrict__ wi) {
    const int l = blockIdx.x;
    __shared__ regrid::Ctl ctl;
    __shared__ double rot[3 * (regrid::kMaxK + 2)];
    __shared__ double fp_slot;
    __shared__ int out_n[3];
    if ((plane_bits[l >> 5] >> (l & 31)) & 1u) {  // all-NaN plane: map_img gives NaN, nothing is fitted
        if (threadIdx.x == 0) {
            nxy[2 * l] = nxy[2 * l + 1] = 0;
            fp[l] = NAN;
            ier[l] = 0;
        }
        return;
    }
    double *txl = tx + (int64_t)l * sl.nxest, *tyl = ty + (int64_t)l * sl.nyest, *cl = c + (int64_t)l * sl.ncmax;
    const regrid::Work w = regrid::carve(wd + (int64_t)l * sl.wd, wi + (int64_t)l * sl.wi, ny, nx, k_rows, k_cols,
                                         sl.nxest, sl.nyest);
    const QuadPlane z{coefq + (int64_t)(l >> 2) * ny * nx * 4 + (l & 3), nx};
    regrid::fit_plane(BlockExec{}, z, ny, nx, k_rows, k_cols, s, sl.nxest, sl.nyest, maxit, txl, tyl, cl, w, ctl, rot,
                      &fp_slot, out_n, fp + l);
    if (threadIdx.x == 0) {
        nxy[2 * l] = out_n[0];
        nxy[2 * l + 1] = out_n[1];
        ier[l] = out_n[2];
    }
}

__global__ void __launch_bounds__(kEvalBlock)
    gather_regrid_kernel(const double *__restrict__ tx, const double *__restrict__ ty, const double *__restrict__ c,
                         const int *__restrict__ nxy, const uint32_t *__restrict__ nanbits,
                         const uint32_t *__restrict__ plane_bits, int n_words, int ny, int nx, int k_rows, int k_cols,
                         RegridSlots sl, int plane_begin, const double *__restrict__ xmap,
                         const double *__restrict__ ymap, int64_t n_cells, uint32_t flags, double *__restrict__ out) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= n_cells) return;
    const int l = plane_begin + blockIdx.y;
    double *dst = out + (int64_t)blockIdx.y * n_cells + cell;
    const double x = __ldg(xmap + cell), y = __ldg(ymap + cell);
    const int word = l >> 5;
    const uint32_t bit = 1u << (l & 31);
    if (isnan(x) || (__ldg(plane_bits + word) & bit)) {  // y is never NaN when x is not (body_xy.py:1697)
        *dst = NAN;
        return;
    }
    if (flags & PM_FLAG_PROPAGATE_NAN) {
        // BodyXY._should_propagate_nan_to_map (body_xy.py:1855-1866)
        if (x < 0.0 || y < 0.0 || x > nx - 1 || y > ny - 1) {
            *dst = NAN;
            return;
        }
        if (__ldg(plane_bits + n_words + word)) {
            const int x0 = max((int)floor(x), 0), x1 = min((int)ceil(x), nx - 1);
            const int y0 = max((int)floor(y), 0), y1 = min((int)ceil(y), ny - 1);
            const uint32_t bad = __ldg(nanbits + ((int64_t)y0 * nx + x0) * n_words + word) |
                                 __ldg(nanbits + ((int64_t)y0 * nx + x1) * n_words + word) |
                                 __ldg(nanbits + ((int64_t)y1 * nx + x0) * n_words + word) |
                                 __ldg(nanbits + ((int64_t)y1 * nx + x1) * n_words + word);
            if (bad & bit) {
                *dst = NAN;
                return;
            }
        }
    }
    // RectBivariateSpline.ev(y, x): FITPACK's x is the image row
    *dst = regrid::evaluate(tx + (int64_t)l * sl.nxest, __ldg(nxy + 2 * l), ty + (int64_t)l * sl.nyest,
                            __ldg(nxy + 2 * l + 1), c + (int64_t)l * sl.ncmax, k_rows, k_cols, y, x);
}

}  // namespace

int64_t regrid_work_bytes(int n_planes, int ny, int nx, int k_rows, int k_cols) {
    const RegridSlots sl = regrid_slots(ny, nx, k_rows, k_cols);
    return (int64_t)n_planes * (sl.wd * (int64_t)sizeof(double) + sl.wi * (int64_t)sizeof(int));
}

cudaError_t launch_regrid_fit(const double *coefq, const uint32_t *plane_bits, int n_planes, int ny, int nx,
                              int k_rows, int k_cols, double s, int maxit, double *tx, double *ty, double *c, int *nxy,
                              double *fp, int *ier, void *work, cudaStream_t st) {
    if (n_planes == 0) return cudaSuccess;
    const RegridSlots sl = regrid_slots(ny, nx, k_rows, k_cols);
    double *wd = static_cast<double *>(work);
    int *wi = reinterpret_cast<int *>(wd + (int64_t)n_planes * sl.wd);
    regrid_fit_kernel<<<n_planes, kFitBlock, 0, st>>>(coefq, plane_bits, ny, nx, k_rows, k_cols, s, maxit, sl, tx, ty,
                                                      c, nxy, fp, ier, wd, wi);
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_gather_regrid(const double *tx, const double *ty, const double *c, const int *nxy,
                                 const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny, int nx,
                                 int k_rows, int k_cols, int plane_begin, int plane_count, const double *xmap,
                                 const double *ymap, int64_t n_cells, uint32_t flags, double *out, cudaStream_t st) {
    if (plane_count == 0 || n_cells == 0) return cudaSuccess;
    const RegridSlots sl = regrid_slots(ny, nx, k_rows, k_cols);
    const int n_words = (n_planes + 31) / 32;
    for (int l0 = 0; l0 < plane_count; l0 += 65535) {  // grid.y limit
        const int nl = plane_count - l0 < 65535 ? plane_count - l0 : 65535;
        dim3 grid((unsigned)((n_cells + kEvalBlock - 1) / kEvalBlock), (unsigned)nl);
        gather_regrid_kernel<<<grid, kEvalBlock, 0, st>>>(tx, ty, c, nxy, nanbits, plane_bits, n_words, ny, nx, k_rows,
                                                          k_cols, sl, plane_begin + l0, xmap, ymap, n_cells, flags,
                                                          out + (int64_t)l0 * n_cells);
        count_launches(1);
    }
    return cudaGetLastError();
}

}  // namespace pm
