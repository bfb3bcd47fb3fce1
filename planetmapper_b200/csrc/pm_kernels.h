// pm_kernels.h - internal launcher declarations shared by the .cu files and capi.cu
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#ifdef PM_TUNING
#include <cstdlib>
#endif

#include "../../include/pm_b200.h"

namespace pm {

constexpr int kBlock = 128;  // threads per CTA for the FP64 geometry kernels

// kernels launched by this library since load (pm_launch_count)
void count_launches(int n);

// Tuning knobs exist only in builds made with -DPM_TUNING (tools/tune_*.py); the product build
// compiles them to their defaults and never reads the environment.
#ifdef PM_TUNING
inline int tune_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v ? atoi(v) : dflt;
}
#else
constexpr int tune_int(const char *, int dflt) { return dflt; }
#endif

cudaError_t launch_backplanes_img(const PMFrame *frames, int n_frames, int nx, int ny, uint64_t mask,
                                  double *out, int sm_count, cudaStream_t st);
cudaError_t launch_backplanes_img_host(const PMFrame *frame_host, int nx, int ny, uint64_t mask, double *out,
                                       int sm_count, cudaStream_t st);
cudaError_t launch_backplanes_points_host(const PMFrame *frame_host, const double *x, const double *y, int64_t n,
                                          uint64_t mask, uint32_t flags, double *out, cudaStream_t st);
cudaError_t launch_backplanes_map(const PMFrame *frames, int n_frames, const double *lon, const double *lat,
                                  int64_t n, uint64_t mask, double *out, int sm_count, cudaStream_t st);
cudaError_t launch_backplanes_map_host(const PMFrame *frame_host, const double *lon, const double *lat, int64_t n,
                                       uint64_t mask, double *out, int sm_count, cudaStream_t st);
cudaError_t launch_xy2lonlat(const PMFrame *frame, const double *x, const double *y, int64_t n, double *lon,
                             double *lat, unsigned long long *n_missed, int sm_count, cudaStream_t st);
cudaError_t launch_lonlat2xy(const PMFrame *frame, const double *lon, const double *lat, int64_t n, double alt,
                             uint32_t flags, double *x, double *y, int sm_count, cudaStream_t st);
cudaError_t launch_transform(const PMFrame *frame, int src, int dst, const double *a, const double *b, int64_t n,
                             double alt, uint32_t flags, const double *aux13_host, double *out_a, double *out_b,
                             unsigned long long *n_missed, cudaStream_t st);
// time-series forms of the three above: frame blockIdx.y, points point_stride doubles apart per frame (0 = shared),
// outputs [n_frames][n], n_missed[n_frames]; aux13: DEVICE [n_frames][13] or NULL
cudaError_t launch_xy2lonlat_batch(const PMFrame *frames, int n_frames, const double *x, const double *y, int64_t n,
                                   int64_t point_stride, double *lon, double *lat, unsigned long long *n_missed,
                                   cudaStream_t st);
cudaError_t launch_lonlat2xy_batch(const PMFrame *frames, int n_frames, const double *lon, const double *lat,
                                   int64_t n, int64_t point_stride, double alt, uint32_t flags, double *x, double *y,
                                   cudaStream_t st);
cudaError_t launch_transform_batch(const PMFrame *frames, int n_frames, int src, int dst, const double *a,
                                   const double *b, int64_t n, int64_t point_stride, double alt, uint32_t flags,
                                   const double *aux13, double *out_a, double *out_b, unsigned long long *n_missed,
                                   cudaStream_t st);
cudaError_t launch_fp64_probe(double *scratch, int kind, int iters, int sm_count, cudaStream_t st);
cudaError_t launch_math_probe(int kind, const double *a, const double *b, int64_t n, double *out,
                              cudaStream_t st);

cudaError_t launch_proj_inverse(int kind, const double *params5, const double *xx, const double *yy,
                                int64_t n, double *lon, double *lat, int sm_count, cudaStream_t st);

cudaError_t launch_proj_forward(int kind, const double *params5, const double *lon, const double *lat, int64_t n,
                                double *xx, double *yy, int sm_count, cudaStream_t st);

cudaError_t launch_gather(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes,
                          int ny, int nx, int plane_begin, int plane_count, const double *xmap, const double *ymap,
                          int64_t n_cells, int64_t cells_per_row, int mode, uint32_t flags, double *out, int sm_count,
                          cudaStream_t st);

// time series: map g serves planes [g * plane_stride, g * plane_stride + planes_per_map); pm_gather_paired is
// planes_per_map = plane_stride = 1
cudaError_t launch_gather_grouped(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes,
                                  int ny, int nx, int n_maps, int planes_per_map, int plane_stride, const double *xmaps,
                                  const double *ymaps, int64_t map_stride, int64_t n_cells, int mode, uint32_t flags,
                                  double *out, int sm_count, cudaStream_t st);

int64_t spline_coef_bytes(int n_planes, int ny, int nx);
int64_t spline_nanbits_bytes(int n_planes, int ny, int nx);
int64_t spline_planebits_bytes(int n_planes);
int64_t spline_work_bytes(int n_planes, int ny, int nx, int degree);
cudaError_t launch_spline_prepare(const double *cube, int n_planes, int ny, int nx, int degree, double *coefq,
                                  uint32_t *nanbits, uint32_t *plane_bits, void *work, int sm_count,
                                  cudaStream_t st);

// map_img with spline_smoothing > 0 (regrid_kernels.cu)
int64_t regrid_work_bytes(int n_planes, int ny, int nx, int k_rows, int k_cols);
cudaError_t launch_regrid_fit(const double *coefq, const uint32_t *plane_bits, int n_planes, int ny, int nx,
                              int k_rows, int k_cols, double s, int maxit, double *tx, double *ty, double *c, int *nxy,
                              double *fp, int *ier, void *work, cudaStream_t st);
cudaError_t launch_gather_regrid(const double *tx, const double *ty, const double *c, const int *nxy,
                                 const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny, int nx,
                                 int k_rows, int k_cols, int plane_begin, int plane_count, const double *xmap,
                                 const double *ymap, int64_t n_cells, uint32_t flags, double *out, cudaStream_t st);

// map_img(interpolation='smooth') (smooth_kernels.cu)
cudaError_t launch_nan_minmax(const double *x, int64_t n, double *out2, cudaStream_t st);
int64_t pchip_work_bytes(int n_planes, int ny, int nx, int n_xs);
cudaError_t launch_pchip_resample(const double *cube, int n_planes, int ny, int nx, int i0, int i1, int j0, int j1,
                                  double x_start, double x_stop, int n_xs, double y_start, double y_stop, int n_ys,
                                  double *fine, void *work, int sm_count, cudaStream_t st);
cudaError_t launch_gather_grid_linear(const double *fine, int n_planes, int n_ys, int n_xs, double x_start,
                                      double x_stop, double y_start, double y_stop, const double *cube, int ny, int nx,
                                      const double *xmap, const double *ymap, int64_t n_cells, uint32_t flags,
                                      double *out, cudaStream_t st);

// FITS data-unit staging (stage_kernels.cu)
cudaError_t launch_fits_stage(const double *const *src, const int64_t *n_elems, const int64_t *dst_offset, int n_units,
                              uint8_t *image, int sm_count, cudaStream_t st);

}  // namespace pm
