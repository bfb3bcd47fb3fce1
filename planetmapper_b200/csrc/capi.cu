// capi.cu - the extern "C" boundary of libpm_b200.so (see include/pm_b200.h).
// Argument checking, device discovery and launch only: no arithmetic lives here.
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>

#include "pm_kernels.h"

namespace pm {
static std::atomic<uint64_t> g_launches{0};
void count_launches(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

static int sm_count() {
    static int cached = 0;
    if (cached > 0) return cached;
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    cached = n;
    return n;
}
static int check(cudaError_t e) {
    if (e == cudaSuccess) return PM_OK;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return PM_ERR_NO_DEVICE;
    std::fprintf(stderr, "libpm_b200: CUDA error: %s\n", cudaGetErrorString(e));
    return PM_ERR_CUDA;
}
}  // namespace pm

using namespace pm;

extern "C" {

int pm_abi_version(void) { return PM_ABI_VERSION; }

const char *pm_error_string(int code) {
    switch (code) {
        case PM_OK: return "ok";
        case PM_ERR_BAD_ARG: return "bad argument";
        case PM_ERR_CUDA: return "CUDA runtime error";
        case PM_ERR_UNSUPPORTED: return "unsupported option";
        case PM_ERR_NO_DEVICE: return "no CUDA device";
        default: return "unknown error";
    }
}

uint64_t pm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int pm_backplanes_img(const PMFrame *frames, int n_frames, int nx, int ny, uint64_t plane_mask, double *out,
                      void *stream) {
    if (!frames || !out || n_frames <= 0 || nx <= 0 || ny <= 0 || n_frames > 65535) return PM_ERR_BAD_ARG;
    plane_mask &= PM_ALL_PLANES;
    if (!plane_mask) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_backplanes_img(frames, n_frames, nx, ny, plane_mask, out, sms, (cudaStream_t)stream));
}

int pm_backplanes_img_host(const PMFrame *frame_host, int nx, int ny, uint64_t plane_mask, double *out, void *stream) {
    if (!frame_host || !out || nx <= 0 || ny <= 0) return PM_ERR_BAD_ARG;
    plane_mask &= PM_ALL_PLANES;
    if (!plane_mask) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_backplanes_img_host(frame_host, nx, ny, plane_mask, out, sms, (cudaStream_t)stream));
}

int pm_backplanes_points_host(const PMFrame *frame_host, const double *x, const double *y, int64_t n,
                              uint64_t plane_mask, uint32_t flags, double *out, void *stream) {
    if (!frame_host || n < 0 || (flags & ~PM_FLAG_RING_ALL)) return PM_ERR_BAD_ARG;
    plane_mask &= PM_ALL_PLANES;
    if (!plane_mask) return PM_ERR_BAD_ARG;
    if (n == 0) return PM_OK;  // empty inputs are valid (and carry null pointers)
    if (!x || !y || !out) return PM_ERR_BAD_ARG;
    if (sm_count() <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_backplanes_points_host(frame_host, x, y, n, plane_mask, flags, out, (cudaStream_t)stream));
}

int pm_backplanes_map(const PMFrame *frame, const double *lon, const double *lat, int64_t n_cells,
                      uint64_t plane_mask, double *out, void *stream) {
    if (!frame || n_cells < 0) return PM_ERR_BAD_ARG;
    plane_mask &= PM_ALL_PLANES;
    if (!plane_mask) return PM_ERR_BAD_ARG;
    if (n_cells == 0) return PM_OK;  // empty inputs are valid (and carry null pointers)
    if (!lon || !lat || !out) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_backplanes_map(frame, 1, lon, lat, n_cells, plane_mask, out, sms, (cudaStream_t)stream));
}

int pm_backplanes_map_host(const PMFrame *frame_host, const double *lon, const double *lat, int64_t n_cells,
                           uint64_t plane_mask, double *out, void *stream) {
    if (!frame_host || n_cells < 0) return PM_ERR_BAD_ARG;
    plane_mask &= PM_ALL_PLANES;
    if (!plane_mask) return PM_ERR_BAD_ARG;
    if (n_cells == 0) return PM_OK;
    if (!lon || !lat || !out) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_backplanes_map_host(frame_host, lon, lat, n_cells, plane_mask, out, sms,
                                            (cudaStream_t)stream));
}

int pm_backplanes_map_batch(const PMFrame *frames, int n_frames, const double *lon, const double *lat,
                            int64_t n_cells, uint64_t plane_mask, double *out, void *stream) {
    if (!frames || n_frames <= 0 || n_frames > 65535 || n_cells < 0) return PM_ERR_BAD_ARG;
    plane_mask &= PM_ALL_PLANES;
    if (!plane_mask) return PM_ERR_BAD_ARG;
    if (n_cells == 0) return PM_OK;
    if (!lon || !lat || !out) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_backplanes_map(frames, n_frames, lon, lat, n_cells, plane_mask, out, sms,
                                       (cudaStream_t)stream));
}

int pm_gather_paired(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny,
                     int nx, const double *xmaps, const double *ymaps, int64_t map_stride, int64_t n_cells, int mode,
                     uint32_t flags, double *out, void *stream) {
    if (n_planes < 0 || ny <= 0 || nx <= 0 || n_cells < 0 || map_stride < n_cells) return PM_ERR_BAD_ARG;
    if (mode != PM_INTERP_NEAREST && mode != PM_INTERP_LINEAR) return PM_ERR_UNSUPPORTED;
    if (n_planes == 0 || n_cells == 0) return PM_OK;
    if (!src || !xmaps || !ymaps || !out) return PM_ERR_BAD_ARG;
    if (mode == PM_INTERP_LINEAR && (!nanbits || !plane_bits || nx < 2 || ny < 2)) return PM_ERR_BAD_ARG;
    if (n_planes > 65535) return PM_ERR_BAD_ARG;
    return check(launch_gather_grouped(src, nanbits, plane_bits, n_planes, ny, nx, n_planes, 1, 1, xmaps, ymaps,
                                       map_stride, n_cells, mode, flags, out, 0, (cudaStream_t)stream));
}

// The sizes, layout and mode of a grouped launch (pm_gather_grouped, pm_composite_grouped): PM_OK or the error.
// `map_len`: the doubles of one epoch's maps, which map_stride must cover; `empty`: nothing to compute
static int grouped_layout(int n_planes, int ny, int nx, int n_maps, int planes_per_map, int plane_stride,
                          int64_t map_stride, int64_t map_len, int64_t n_cells, int mode, bool &empty) {
    if (n_planes < 0 || ny <= 0 || nx <= 0 || n_maps < 0 || n_maps > 65535 || planes_per_map < 0 ||
        plane_stride < planes_per_map || n_cells < 0 || map_stride < map_len)
        return PM_ERR_BAD_ARG;
    empty = n_maps == 0 || planes_per_map == 0 || n_cells == 0;  // valid, with null pointers
    if (!empty && (int64_t)(n_maps - 1) * plane_stride + planes_per_map > n_planes) return PM_ERR_BAD_ARG;
    if (!empty && map_stride > INT64_MAX / n_maps) return PM_ERR_BAD_ARG;
    int ky, kx;
    if (interp_degrees(mode, ky, kx) != PM_OK) return PM_ERR_UNSUPPORTED;
    return nx <= kx || ny <= ky ? PM_ERR_BAD_ARG : PM_OK;
}

int pm_gather_grouped(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny,
                      int nx, int n_maps, int planes_per_map, int plane_stride, const double *xmaps,
                      const double *ymaps, int64_t map_stride, int64_t n_cells, int mode, uint32_t flags, double *out,
                      void *stream) {
    bool empty = true;
    const int rc = grouped_layout(n_planes, ny, nx, n_maps, planes_per_map, plane_stride, map_stride, n_cells, n_cells,
                                  mode, empty);
    if (rc != PM_OK) return rc;
    if (empty) return PM_OK;
    if (!src || !xmaps || !ymaps || !out) return PM_ERR_BAD_ARG;
    if (mode != PM_INTERP_NEAREST && (!nanbits || !plane_bits)) return PM_ERR_BAD_ARG;
    if (planes_per_map > 65535 * 128) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_gather_grouped(src, nanbits, plane_bits, n_planes, ny, nx, n_maps, planes_per_map,
                                       plane_stride, xmaps, ymaps, map_stride, n_cells, mode, flags, out, sms,
                                       (cudaStream_t)stream));
}

int pm_composite_grouped(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny,
                         int nx, int n_maps, int planes_per_map, int plane_stride, const double *maps, int n_map_planes,
                         int64_t map_stride, int64_t n_cells, int mode, uint32_t flags, int method,
                         double max_emission, int epoch_begin, int first, int last, double *value, double *key,
                         int32_t *tag, void *stream) {
    if (method != PM_COMPOSITE_MEAN && method != PM_COMPOSITE_MIN_EMISSION) return PM_ERR_UNSUPPORTED;
    if (n_map_planes != 2 && n_map_planes != 3) return PM_ERR_BAD_ARG;
    // without an EMISSION plane there is nothing to cut on or to rank by
    if (n_map_planes == 2 && (method != PM_COMPOSITE_MEAN || max_emission != INFINITY)) return PM_ERR_BAD_ARG;
    if (max_emission != max_emission || (flags & ~PM_FLAG_PROPAGATE_NAN) || (first & ~1) || (last & ~1) ||
        epoch_begin < 0 || (int64_t)epoch_begin + n_maps > INT32_MAX)
        return PM_ERR_BAD_ARG;
    bool empty = true;
    const int rc = grouped_layout(n_planes, ny, nx, n_maps, planes_per_map, plane_stride, map_stride,
                                  (int64_t)n_map_planes * n_cells, n_cells, mode, empty);
    if (rc != PM_OK) return rc;
    if (empty) return PM_OK;
    if (!src || !maps || !value || !tag || (method == PM_COMPOSITE_MIN_EMISSION && !key)) return PM_ERR_BAD_ARG;
    if (mode != PM_INTERP_NEAREST && (!nanbits || !plane_bits)) return PM_ERR_BAD_ARG;
    if (planes_per_map > 65535 * 4) return PM_ERR_BAD_ARG;   // plane groups of four along gridDim.y
    if (sm_count() <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_composite_grouped(src, nanbits, plane_bits, n_planes, ny, nx, n_maps, planes_per_map,
                                          plane_stride, maps, n_map_planes, map_stride, n_cells, mode, flags, method,
                                          max_emission, epoch_begin, first != 0, last != 0, value, key, tag,
                                          (cudaStream_t)stream));
}

int pm_xy2lonlat(const PMFrame *frame, const double *x, const double *y, int64_t n, double *lon, double *lat,
                 int64_t *n_missed, void *stream) {
    if (!frame || n < 0) return PM_ERR_BAD_ARG;
    if (n == 0) return PM_OK;
    if (!x || !y || !lon || !lat) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_xy2lonlat(frame, x, y, n, lon, lat, (unsigned long long *)n_missed, sms,
                                  (cudaStream_t)stream));
}

int pm_lonlat2xy_alt(const PMFrame *frame, const double *lon, const double *lat, int64_t n, double alt,
                     uint32_t flags, double *x, double *y, void *stream) {
    if (!frame || n < 0 || !(alt == alt)) return PM_ERR_BAD_ARG;
    if (n == 0) return PM_OK;
    if (!x || !y || !lon || !lat) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_lonlat2xy(frame, lon, lat, n, alt, flags, x, y, sms, (cudaStream_t)stream));
}
int pm_lonlat2xy(const PMFrame *frame, const double *lon, const double *lat, int64_t n, uint32_t flags,
                 double *x, double *y, void *stream) {
    return pm_lonlat2xy_alt(frame, lon, lat, n, 0.0, flags, x, y, stream);
}

int pm_transform(const PMFrame *frame, int src, int dst, const double *a, const double *b, int64_t n, double alt,
                 uint32_t flags, const double *aux13_host, double *out_a, double *out_b, int64_t *n_missed,
                 void *stream) {
    if (!frame || n < 0 || !(alt == alt)) return PM_ERR_BAD_ARG;
    if (src < PM_COORD_XY || src > PM_COORD_LONLAT || dst < PM_COORD_XY || dst > PM_COORD_CENTRIC) return PM_ERR_BAD_ARG;
    if ((src == dst && src != PM_COORD_LONLAT) || (dst == PM_COORD_CENTRIC && src == PM_COORD_CENTRIC))
        return PM_ERR_UNSUPPORTED;
    if (n == 0) return PM_OK;
    if (!a || !b || !out_a || !out_b) return PM_ERR_BAD_ARG;
    if (sm_count() <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_transform(frame, src, dst, a, b, n, alt, flags, aux13_host, out_a, out_b,
                                  (unsigned long long *)n_missed, (cudaStream_t)stream));
}

// The time-series entry points check every argument before touching the device
static bool batch_ok(const PMFrame *frames, int n_frames, int64_t n, int64_t point_stride) {
    return frames && n_frames > 0 && n_frames <= 65535 && n >= 0 && (point_stride == 0 || point_stride >= n) &&
           point_stride <= INT64_MAX / 65535;
}
static bool finite_alt(double alt) { return alt - alt == 0.0; }
static bool coords_ok(int src, int dst) {
    return src >= PM_COORD_XY && src <= PM_COORD_LONLAT && dst >= PM_COORD_XY && dst <= PM_COORD_CENTRIC;
}

int pm_xy2lonlat_batch(const PMFrame *frames, int n_frames, const double *x, const double *y, int64_t n,
                       int64_t point_stride, double *lon, double *lat, int64_t *n_missed, void *stream) {
    if (!batch_ok(frames, n_frames, n, point_stride)) return PM_ERR_BAD_ARG;
    if (n == 0) return PM_OK;
    if (!x || !y || !lon || !lat) return PM_ERR_BAD_ARG;
    if (sm_count() <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_xy2lonlat_batch(frames, n_frames, x, y, n, point_stride, lon, lat,
                                        (unsigned long long *)n_missed, (cudaStream_t)stream));
}

int pm_lonlat2xy_batch(const PMFrame *frames, int n_frames, const double *lon, const double *lat, int64_t n,
                       int64_t point_stride, double alt, uint32_t flags, double *x, double *y, void *stream) {
    if (!batch_ok(frames, n_frames, n, point_stride) || !finite_alt(alt)) return PM_ERR_BAD_ARG;
    if (flags & ~(PM_FLAG_NOT_VISIBLE_NAN | PM_FLAG_PLANETOCENTRIC)) return PM_ERR_BAD_ARG;
    if (n == 0) return PM_OK;
    if (!lon || !lat || !x || !y) return PM_ERR_BAD_ARG;
    if (sm_count() <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_lonlat2xy_batch(frames, n_frames, lon, lat, n, point_stride, alt, flags, x, y,
                                        (cudaStream_t)stream));
}

int pm_transform_batch(const PMFrame *frames, int n_frames, int src, int dst, const double *a, const double *b,
                       int64_t n, int64_t point_stride, double alt, uint32_t flags, const double *aux13,
                       double *out_a, double *out_b, int64_t *n_missed, void *stream) {
    if (!batch_ok(frames, n_frames, n, point_stride) || !finite_alt(alt) || !coords_ok(src, dst)) return PM_ERR_BAD_ARG;
    if (flags & ~(PM_FLAG_NOT_VISIBLE_NAN | PM_FLAG_PLANETOCENTRIC)) return PM_ERR_BAD_ARG;
    if (src == dst && src != PM_COORD_LONLAT) return PM_ERR_UNSUPPORTED;
    if (n == 0) return PM_OK;
    if (!a || !b || !out_a || !out_b) return PM_ERR_BAD_ARG;
    if (sm_count() <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_transform_batch(frames, n_frames, src, dst, a, b, n, point_stride, alt, flags, aux13, out_a,
                                        out_b, (unsigned long long *)n_missed, (cudaStream_t)stream));
}

int pm_proj_inverse(int kind, const double *params5_host, const double *xx, const double *yy, int64_t n,
                    double *lon, double *lat, void *stream) {
    if (!params5_host || n < 0) return PM_ERR_BAD_ARG;
    if (kind < PM_PROJ_ORTHOGRAPHIC || kind > PM_PROJ_AZIMUTHAL_EQUAL_AREA) return PM_ERR_UNSUPPORTED;
    if (n == 0) return PM_OK;
    if (!xx || !yy || !lon || !lat) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_proj_inverse(kind, params5_host, xx, yy, n, lon, lat, sms, (cudaStream_t)stream));
}

int pm_proj_forward(int kind, const double *params5_host, const double *lon, const double *lat, int64_t n,
                    double *xx, double *yy, void *stream) {
    if (!params5_host || n < 0) return PM_ERR_BAD_ARG;
    if (kind < PM_PROJ_ORTHOGRAPHIC || kind > PM_PROJ_AZIMUTHAL_EQUAL_AREA) return PM_ERR_UNSUPPORTED;
    if (n == 0) return PM_OK;
    if (!xx || !yy || !lon || !lat) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_proj_forward(kind, params5_host, lon, lat, n, xx, yy, sms, (cudaStream_t)stream));
}

int pm_gather(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny, int nx,
              int plane_begin, int plane_count, const double *xmap, const double *ymap, int64_t n_cells,
              int64_t cells_per_row, int mode, uint32_t flags, double *out, void *stream) {
    if (n_planes < 0 || ny <= 0 || nx <= 0 || n_cells < 0 || plane_begin < 0 || plane_count < 0 ||
        plane_begin + plane_count > n_planes)
        return PM_ERR_BAD_ARG;
    const bool empty = n_cells == 0 || plane_count == 0;  // valid, and the empty arrays carry null pointers
    if (!empty && (!src || !xmap || !ymap || !out)) return PM_ERR_BAD_ARG;
    int ky, kx;
    if (interp_degrees(mode, ky, kx) != PM_OK) return PM_ERR_UNSUPPORTED;
    if (nx <= kx || ny <= ky) return PM_ERR_BAD_ARG;
    if (empty) return PM_OK;
    if (mode != PM_INTERP_NEAREST && (!nanbits || !plane_bits || (plane_begin & 3))) return PM_ERR_BAD_ARG;
    if (plane_count > 65535 * 128) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_gather(src, nanbits, plane_bits, n_planes, ny, nx, plane_begin, plane_count, xmap, ymap,
                               n_cells, cells_per_row, mode, flags, out, sms, (cudaStream_t)stream));
}

int64_t pm_spline_coef_bytes(int n_planes, int ny, int nx) {
    if (n_planes < 0 || ny <= 0 || nx <= 0) return PM_ERR_BAD_ARG;
    return spline_coef_bytes(n_planes, ny, nx);
}
int64_t pm_spline_nanbits_bytes(int n_planes, int ny, int nx) {
    if (n_planes < 0 || ny <= 0 || nx <= 0) return PM_ERR_BAD_ARG;
    return spline_nanbits_bytes(n_planes, ny, nx);
}
int64_t pm_spline_planebits_bytes(int n_planes) {
    if (n_planes < 0) return PM_ERR_BAD_ARG;
    return spline_planebits_bytes(n_planes);
}
int64_t pm_spline_work_bytes(int n_planes, int ny, int nx, int degree) {
    if (n_planes < 0 || ny <= 0 || nx <= 0) return PM_ERR_BAD_ARG;
    return spline_work_bytes(n_planes, ny, nx, degree);
}

int pm_spline_prepare(const double *cube, int n_planes, int ny, int nx, int degree, double *coef,
                      uint32_t *nanbits, uint32_t *plane_bits, void *work, void *stream) {
    if (!cube || !coef || !nanbits || !plane_bits || !work || n_planes < 0 || ny <= 0 || nx <= 0)
        return PM_ERR_BAD_ARG;
    int ky, kx;
    if (interp_degrees(degree, ky, kx) != PM_OK || ky == 0) return PM_ERR_UNSUPPORTED;   // nearest needs no spline
    if (nx <= kx || ny <= ky) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_spline_prepare(cube, n_planes, ny, nx, degree, coef, nanbits, plane_bits, work, sms,
                                       (cudaStream_t)stream));
}

int pm_nan_minmax(const double *x, int64_t n, double *out2, void *stream) {
    if (!x || !out2 || n <= 0) return PM_ERR_BAD_ARG;
    return check(launch_nan_minmax(x, n, out2, (cudaStream_t)stream));
}

int64_t pm_pchip_work_bytes(int n_planes, int ny, int nx, int n_xs) {
    if (n_planes < 0 || ny <= 0 || nx <= 0 || n_xs <= 0) return PM_ERR_BAD_ARG;
    return pchip_work_bytes(n_planes, ny, nx, n_xs);
}

int pm_pchip_resample(const double *cube, int n_planes, int ny, int nx, int x_first, int x_last, int y_first,
                      int y_last, int n_xs, int n_ys, double *fine, void *work, void *stream) {
    if (!cube || !fine || !work || n_planes < 0 || ny <= 0 || nx <= 0 || n_xs < 1 || n_ys < 1 || x_first < 0 ||
        x_last >= nx || x_first > x_last || y_first < 0 || y_last >= ny || y_first > y_last)
        return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_pchip_resample(cube, n_planes, ny, nx, x_first, x_last, y_first, y_last, (double)x_first,
                                       (double)x_last, n_xs, (double)y_first, (double)y_last, n_ys, fine, work, sms,
                                       (cudaStream_t)stream));
}

static bool regrid_degrees_ok(int k_rows, int k_cols) { return k_rows >= 1 && k_rows <= 3 && k_cols >= 1 && k_cols <= 3; }

int64_t pm_regrid_work_bytes(int n_planes, int ny, int nx, int k_rows, int k_cols) {
    if (n_planes < 0 || ny <= 0 || nx <= 0) return PM_ERR_BAD_ARG;
    if (!regrid_degrees_ok(k_rows, k_cols)) return PM_ERR_UNSUPPORTED;
    return regrid_work_bytes(n_planes, ny, nx, k_rows, k_cols);
}

int pm_regrid_fit(const double *coef, const uint32_t *plane_bits, int n_planes, int ny, int nx, int k_rows,
                  int k_cols, double s, int maxit, double *tx, double *ty, double *c, int *nxy, double *fp, int *ier,
                  void *work, void *stream) {
    if (n_planes < 0 || ny <= 0 || nx <= 0 || !(s > 0.0) || !(s <= 1.79769313486231570e308) || maxit < 1)
        return PM_ERR_BAD_ARG;
    if (!regrid_degrees_ok(k_rows, k_cols)) return PM_ERR_UNSUPPORTED;
    if (ny <= k_rows || nx <= k_cols) return PM_ERR_BAD_ARG;
    if (n_planes == 0) return PM_OK;
    if (!coef || !plane_bits || !tx || !ty || !c || !nxy || !fp || !ier || !work) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_regrid_fit(coef, plane_bits, n_planes, ny, nx, k_rows, k_cols, s, maxit, tx, ty, c, nxy, fp,
                                   ier, work, (cudaStream_t)stream));
}

int pm_gather_regrid(const double *tx, const double *ty, const double *c, const int *nxy, const uint32_t *nanbits,
                     const uint32_t *plane_bits, int n_planes, int ny, int nx, int k_rows, int k_cols, int plane_begin,
                     int plane_count, const double *xmap, const double *ymap, int64_t n_cells, uint32_t flags,
                     double *out, void *stream) {
    if (n_planes < 0 || ny <= 0 || nx <= 0 || n_cells < 0 || plane_begin < 0 || plane_count < 0 ||
        plane_begin > n_planes - plane_count || (flags & ~PM_FLAG_PROPAGATE_NAN))
        return PM_ERR_BAD_ARG;
    if (!regrid_degrees_ok(k_rows, k_cols)) return PM_ERR_UNSUPPORTED;
    if (ny <= k_rows || nx <= k_cols) return PM_ERR_BAD_ARG;
    if (n_cells == 0 || plane_count == 0) return PM_OK;  // the empty arrays may carry null pointers
    if (!tx || !ty || !c || !nxy || !nanbits || !plane_bits || !xmap || !ymap || !out) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_gather_regrid(tx, ty, c, nxy, nanbits, plane_bits, n_planes, ny, nx, k_rows, k_cols,
                                      plane_begin, plane_count, xmap, ymap, n_cells, flags, out, (cudaStream_t)stream));
}

int pm_gather_grid_linear(const double *fine, int n_planes, int n_ys, int n_xs, int x_first, int x_last, int y_first,
                          int y_last, const double *cube, int ny, int nx, const double *xmap, const double *ymap,
                          int64_t n_cells, uint32_t flags, double *out, void *stream) {
    if (!fine || !cube || !xmap || !ymap || !out || n_planes < 0 || n_ys < 1 || n_xs < 1 || ny <= 0 || nx <= 0 ||
        n_cells < 0)
        return PM_ERR_BAD_ARG;
    return check(launch_gather_grid_linear(fine, n_planes, n_ys, n_xs, (double)x_first, (double)x_last, (double)y_first,
                                           (double)y_last, cube, ny, nx, xmap, ymap, n_cells, flags, out,
                                           (cudaStream_t)stream));
}

int64_t pm_fits_data_unit_bytes(int64_t n_elems) {
    if (n_elems < 0) return PM_ERR_BAD_ARG;
    return (n_elems * 8 + 2879) / 2880 * 2880;
}

int pm_fits_stage(const double *const *src, const int64_t *n_elems, const int64_t *dst_offset, int n_units,
                  uint8_t *image, void *stream) {
    if (n_units < 0 || (n_units > 0 && (!src || !n_elems || !dst_offset || !image))) return PM_ERR_BAD_ARG;
    for (int u = 0; u < n_units; u++)
        if (n_elems[u] < 0 || dst_offset[u] < 0 || (dst_offset[u] & 7) || (n_elems[u] > 0 && !src[u]))
            return PM_ERR_BAD_ARG;
    if (n_units == 0) return PM_OK;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    return check(launch_fits_stage(src, n_elems, dst_offset, n_units, image, sms, (cudaStream_t)stream));
}

int pm_math_probe(int kind, const double *a, const double *b, int64_t n, double *out, void *stream) {
    if (!a || !out || n < 0 || kind < 0 || kind > 13) return PM_ERR_BAD_ARG;
    if ((kind == 5 || kind == 7 || kind == 10 || kind == 11) && !b) return PM_ERR_BAD_ARG;
    if (n == 0) return PM_OK;
    return check(launch_math_probe(kind, a, b, n, out, (cudaStream_t)stream));
}

int pm_fp64_probe(int kind, int iters, double *ms_host, double *flops_host) {
    if (iters <= 0 || !ms_host || !flops_host || kind < 0 || kind > 1) return PM_ERR_BAD_ARG;
    int sms = sm_count();
    if (sms <= 0) return PM_ERR_NO_DEVICE;
    double *scratch = nullptr;
    if (cudaMalloc(&scratch, 65 * sizeof(double)) != cudaSuccess) return PM_ERR_CUDA;
    double init[65];
    for (int i = 0; i < 65; i++) init[i] = 0.999 + 1e-5 * i;
    cudaMemcpy(scratch, init, sizeof(init), cudaMemcpyHostToDevice);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    launch_fp64_probe(scratch, kind, iters, sms, 0);  // warm-up
    cudaDeviceSynchronize();
    cudaEventRecord(e0, 0);
    cudaError_t err = launch_fp64_probe(scratch, kind, iters, sms, 0);
    cudaEventRecord(e1, 0);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(scratch);
    *ms_host = (double)ms;
    // 8 independent FMA chains per thread, 2 flop per FMA
    *flops_host = 2.0 * 8.0 * (double)iters * 256.0 * (double)sms * 8.0;
    return check(err);
}
int pm_fp64_peak_probe(int iters, double *ms_host, double *flops_host) {
    return pm_fp64_probe(0, iters, ms_host, flops_host);
}

}  // extern "C"
