/*
 * pm_b200.h - C ABI of the B200-native PlanetMapper hot path (libpm_b200.so).
 *
 * The reference (ortk95/planetmapper, pure Python) has no FFI of its own: its
 * per-pixel work is a Python loop making one ctypes CSPICE call per pixel per
 * stage.  The entry points below are what a maintainer would bind (ctypes stub in
 * INTEGRATION.md) to replace those loops; each cites the reference method it
 * replaces.  Plain pointers and sizes only; every function returns PM_OK (0) or a
 * negative PM_ERR_* code, writes NaN for invalid pixels / cells and never throws.
 *
 * All `double*` data arguments are DEVICE pointers unless the name ends in
 * `_host`.  `stream` is a cudaStream_t passed as void* (NULL = default stream).
 * Work is enqueued asynchronously on `stream`; the caller synchronises.
 */
#ifndef PM_B200_H
#define PM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PM_OK 0
#define PM_ERR_BAD_ARG (-1)
#define PM_ERR_CUDA (-2)
#define PM_ERR_UNSUPPORTED (-3)
#define PM_ERR_NO_DEVICE (-4)

#define PM_ABI_VERSION 10

/*
 * Per-frame constants, computed once per frame on the host from SPICE
 * (planetmapper/base.py:815-837, planetmapper/body.py:522-588,
 * planetmapper/body_xy.py:355-373).  All doubles, so the struct is also a flat
 * double[PM_FRAME_NDOUBLES]; the Python packer is planetmapper_b200/frame.py.
 * Vectors are J2000 unless stated; "body" = target body-fixed frame (IAU_*).
 */
typedef struct PMFrame {
    double et;          /* observation epoch, TDB s past J2000 (Body.et)              */
    double clight;      /* km/s                                                        */
    double lt0;         /* light time to target centre (Body.target_light_time)       */
    double t_ref;       /* et - lt0: reference epoch for the linear models below      */
    double P0[3];       /* observer -> target centre at t_ref (Body._target_obsvec)   */
    double VT[3];       /* target centre SSB velocity at t_ref                        */
    double AT[3];       /* target centre SSB acceleration at t_ref                    */
    double VO[3];       /* observer SSB velocity at et                                */
    double S0[3];       /* Sun(t_ref - lts0) - target centre(t_ref)                   */
    double VS[3];       /* Sun SSB velocity at t_ref - lts0                           */
    double lts0;        /* Sun -> target centre light time at t_ref                   */
    double R0[9];       /* J2000 -> body rotation at t_ref, row-major                 */
    double omega[3];    /* body-frame angular velocity, dR/dt = -[omega]x R (rad/s)   */
    double radii[3];    /* ellipsoid radii incl. any altitude adjustment (km)         */
    double re;          /* spheroid equatorial radius used by recpgr/pgrrec           */
    double f;           /* spheroid flattening used by recpgr/pgrrec                  */
    double lon_sign;    /* +1 planetographic east-positive, -1 west-positive          */
    double prograde;    /* 1 prograde, 0 retrograde (et2lst)                          */
    double sub_t[3];    /* sub-observer point, body (Body._subpoint_targvec)          */
    double sub_ray[3];  /* observer -> sub-point, body (Body._subpoint_rayvec)        */
    double sub_obs[3];  /* same, J2000 (Body._subpoint_obsvec)                        */
    double sub_dt;      /* Body._subpoint_et - t_ref                                  */
    double sub_dist;    /* Body.subpoint_distance                                     */
    double ring_n[3];   /* ring plane unit normal (Body._ring_plane)                  */
    double ring_c;      /* ring plane constant, >= 0                                  */
    double sun_lon_lst; /* body-fixed planetocentric Sun longitude used by et2lst     */
    double M[9];        /* obsvec -> angular rotation (body.py:1318-1343), row-major  */
    double ang2km[4];   /* angular(arcsec) -> km 2x2 (body.py:1636-1639)              */
    double km_per_arcsec;
    double A[6];        /* xy -> angular arcsec, rows [a00 a01 a02],[a10 a11 a12]     */
    double Ainv[6];     /* angular arcsec -> xy                                       */
    double nx, ny;      /* image size (integers stored as doubles)                    */
    double x0, y0;      /* disc centre (pixels)                                       */
    double r_cut2;      /* squared early-out radius (body_xy.py:3201-3203)            */
    double optimize_speed; /* 1 = apply the early-out (SpiceBase._optimize_speed)     */
    double r_eq;        /* equatorial radius used for RING-RADIUS = alt + r_eq        */
    double reserved[1];
} PMFrame;

#define PM_FRAME_NDOUBLES 92

/* Backplane ids = registration order in BodyXY._register_default_backplanes
 * (planetmapper/body_xy.py:4198-4356). A plane mask has bit `id` set. */
enum PMPlane {
    PM_LON_GRAPHIC = 0, PM_LAT_GRAPHIC = 1, PM_LON_CENTRIC = 2, PM_LAT_CENTRIC = 3,
    PM_RA = 4, PM_DEC = 5, PM_PIXEL_X = 6, PM_PIXEL_Y = 7, PM_KM_X = 8, PM_KM_Y = 9,
    PM_ANGULAR_X = 10, PM_ANGULAR_Y = 11, PM_PHASE = 12, PM_INCIDENCE = 13,
    PM_EMISSION = 14, PM_AZIMUTH = 15, PM_LOCAL_SOLAR_TIME = 16, PM_DISTANCE = 17,
    PM_RADIAL_VELOCITY = 18, PM_DOPPLER = 19, PM_LIMB_DISTANCE = 20,
    PM_LIMB_LON_GRAPHIC = 21, PM_LIMB_LAT_GRAPHIC = 22, PM_RING_RADIUS = 23,
    PM_RING_LON_GRAPHIC = 24, PM_RING_DISTANCE = 25, PM_N_PLANES = 26
};
#define PM_ALL_PLANES ((1ull << PM_N_PLANES) - 1ull)

/* interpolation modes of pm_gather (BodyXY.map_img, body_xy.py:1414-1631) */
#define PM_INTERP_NEAREST 0
#define PM_INTERP_LINEAR 1
#define PM_INTERP_QUADRATIC 2
#define PM_INTERP_CUBIC 3
/* mixed spline degrees, RectBivariateSpline(kx = ky_rows, ky = kx_cols): degree along image
 * rows (y) in bits 4-7, along columns (x) in bits 0-3, each 1..3 */
#define PM_INTERP_MIXED 0x100
#define PM_INTERP_MIXED_MODE(deg_rows, deg_cols) (PM_INTERP_MIXED | ((deg_rows) << 4) | (deg_cols))

/* projection kinds of pm_proj_inverse (BodyXY.generate_map_coordinates,
 * body_xy.py:2899-2969) */
#define PM_PROJ_ORTHOGRAPHIC 1
#define PM_PROJ_AZIMUTHAL 2
#define PM_PROJ_AZIMUTHAL_EQUAL_AREA 3

/* flags */
#define PM_FLAG_NOT_VISIBLE_NAN 1u /* lonlat2xy(not_visible_nan=True)               */
#define PM_FLAG_PROPAGATE_NAN 2u   /* map_img(propagate_nan=True)                   */
#define PM_FLAG_PLANETOCENTRIC 4u   /* lonlat2xy(planetocentric=True) inputs         */
#define PM_FLAG_RING_ALL 8u         /* ring_plane_coordinates(only_visible=False)    */

/* coordinate systems of pm_transform (the five systems of Body / BodyXY, planetmapper/body.py:1083-1900,
 * planetmapper/body_xy.py:385-676; CENTRIC = planetocentric lon / lat as a destination) */
#define PM_COORD_XY 0
#define PM_COORD_ANGULAR 1
#define PM_COORD_KM 2
#define PM_COORD_RADEC 3
#define PM_COORD_LONLAT 4
#define PM_COORD_CENTRIC 5

int pm_abi_version(void);
const char *pm_error_string(int code);
/* number of CUDA kernels this library has launched since load (bench evidence) */
uint64_t pm_launch_count(void);

/*
 * Image-direction backplanes: replaces the per-pixel loops
 * BodyXY._get_targvec_img (body_xy.py:3197), _get_lonlat_img (:3284),
 * _get_lonlat_centric_img (:3349), _get_radec_img (:3413), _get_km_xy_img (:3547),
 * _get_illumination_gie_img (:3661), get_azimuth_angle_img (:3744),
 * get_local_solar_time_img (:3790), _get_state_imgs (:3832),
 * get_radial_velocity_img (:3898), get_doppler_img (:3938),
 * _get_limb_coordinate_imgs (:3967), _get_ring_plane_coordinate_imgs (:4061).
 * `frames`: n_frames PMFrame structs in DEVICE memory (all with the same nx, ny).
 * `out`: [n_frames][popcount(mask)][ny][nx] doubles, planes in increasing id order.
 */
int pm_backplanes_img(const PMFrame *frames, int n_frames, int nx, int ny,
                      uint64_t plane_mask, double *out, void *stream);
/* The same for ONE frame whose constants are in HOST memory (the usual case: the host has just
 * computed them - BodyXY's constructor and setters, planetmapper/body_xy.py:186-232, :696-961).
 * The 92 constants and the values derived from them travel with the launch as a kernel parameter,
 * so the per-pixel code reads them from the constant bank; no host -> device copy is enqueued.
 * `out` is a DEVICE pointer: [popcount(mask)][ny][nx]. */
int pm_backplanes_img_host(const PMFrame *frame_host, int nx, int ny, uint64_t plane_mask,
                           double *out, void *stream);
/* Image-direction backplanes at n arbitrary image positions (x[i], y[i]) - fractional, outside the
 * image, in any order - of ONE frame given in HOST memory (constants as a kernel parameter, like
 * pm_backplanes_img_host): the per-point geometry queries of Body (illumination / limb / ring-plane
 * coordinates at a direction, planetmapper/body.py:2081-2110, :2577-2615).  `x`, `y`, `out` are
 * DEVICE pointers; out: [popcount(mask)][n].  At integer (x, y) every plane equals
 * pm_backplanes_img_host's pixel bit for bit.  A point whose x or y is not finite gets NaN in every
 * plane but PIXEL-X / PIXEL-Y, which echo the input.  flags: 0 or PM_FLAG_RING_ALL = ring-plane
 * coordinates without the "hidden behind the body" test (Body.ring_plane_coordinates with
 * only_visible=False).  n = 0 is valid with NULL pointers. */
int pm_backplanes_points_host(const PMFrame *frame_host, const double *x, const double *y, int64_t n,
                              uint64_t plane_mask, uint32_t flags, double *out, void *stream);

/*
 * Map-direction backplanes on arbitrary lon/lat cells (degrees, planetographic):
 * replaces _get_targvec_map (body_xy.py:3230), _get_illumf_map (:3671),
 * _get_obsvec_map (:3275), _get_radec_map (:3423), _get_xy_map (:3482),
 * _get_km_xy_map (:3557), _get_lonlat_centric_map (:3357), _get_state_maps (:3851),
 * get_radial_velocity_map (:3917), get_local_solar_time_map (:3812),
 * _get_limb_coordinate_maps (:3980), _get_ring_plane_coordinate_maps (:4090).
 * PIXEL-X / PIXEL-Y are x_map / y_map.  `out`: [popcount(mask)][n_cells].
 */
int pm_backplanes_map(const PMFrame *frame, const double *lon, const double *lat,
                      int64_t n_cells, uint64_t plane_mask, double *out, void *stream);
/* The same for ONE frame whose constants are in HOST memory (see pm_backplanes_img_host): this is what
 * BodyXY.get_backplane_map and the x / y map of BodyXY.map_img (body_xy.py:1414, :3482) launch.  `lon`,
 * `lat`, `out` are DEVICE pointers.  With plane_mask = PIXEL-X | PIXEL-Y the kernel is the instantiation
 * that computes only what x_map / y_map need (illumf's emission angle for the visibility test). */
int pm_backplanes_map_host(const PMFrame *frame_host, const double *lon, const double *lat,
                           int64_t n_cells, uint64_t plane_mask, double *out, void *stream);

/*
 * Time series (BASELINE config C5: a fresh BodyXY per epoch, then map_img of that epoch's image,
 * i.e. body_xy.py:3482-3491 + :1414-1631 once per frame in the reference).
 *   pm_backplanes_map_batch  pm_backplanes_map for n_frames frames sharing one lon / lat grid, one
 *                            launch; out: [n_frames][popcount(mask)][n_cells].
 *   pm_gather_paired         map_img where plane l of the cube is mapped with ITS OWN x / y map
 *                            (xmaps + l * map_stride): nearest (src = the cube as is) or linear
 *                            (src / nanbits / plane_bits = pm_spline_prepare(degree 1) outputs);
 *                            out: [n_planes][n_cells].  Same arithmetic per cell as pm_gather.
 *   pm_gather_grouped        map_img / get_mapped_data of one image or cube per epoch: map g (xmaps +
 *                            g * map_stride, g < n_maps <= 65535) serves planes [g * plane_stride,
 *                            g * plane_stride + planes_per_map) of an n_planes cube, with every mode of
 *                            pm_gather (nearest: `src` = the raw cube; spline modes: pm_spline_prepare's
 *                            three buffers for the whole cube).  out: [n_maps][planes_per_map][n_cells].
 *                            Group g equals pm_gather of its planes through map g bit for bit, except a
 *                            cubic group of one plane on a map of >= 20 cells per image pixel, whose sums
 *                            differ from pm_gather's DMMA order in the last bits.  A plane_stride that is a
 *                            multiple of 4 (groups start on a plane quad) is the fast layout for
 *                            planes_per_map > 1; pm_gather_paired is planes_per_map = plane_stride = 1.
 *                            Empty input (n_maps, planes_per_map or n_cells 0) is valid with NULL pointers.
 */
int pm_backplanes_map_batch(const PMFrame *frames, int n_frames, const double *lon, const double *lat,
                            int64_t n_cells, uint64_t plane_mask, double *out, void *stream);
int pm_gather_paired(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits,
                     int n_planes, int ny, int nx, const double *xmaps, const double *ymaps,
                     int64_t map_stride, int64_t n_cells, int mode, uint32_t flags, double *out,
                     void *stream);
int pm_gather_grouped(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits,
                      int n_planes, int ny, int nx, int n_maps, int planes_per_map, int plane_stride,
                      const double *xmaps, const double *ymaps, int64_t map_stride, int64_t n_cells,
                      int mode, uint32_t flags, double *out, void *stream);

/*
 * Vectorised point transforms: replace SpiceBase._maybe_transform_as_arrays
 * (base.py:718-757) driving BodyXY._xy2lonlat (body_xy.py:482) and _lonlat2xy (:544).
 * Misses / invisible points produce NaN; `n_missed` (device int64, may be NULL)
 * counts xy2lonlat rays that missed the body (the host raises NotFoundError when
 * not_found_nan=False, body.py:1073-1078).
 */
int pm_xy2lonlat(const PMFrame *frame, const double *x, const double *y, int64_t n,
                 double *lon, double *lat, int64_t *n_missed, void *stream);
int pm_lonlat2xy(const PMFrame *frame, const double *lon, const double *lat, int64_t n,
                 uint32_t flags, double *x, double *y, void *stream);
/* Same with a point altitude (km above the spheroid, pgrrec's `alt`): for alt != 0 the
 * visibility test is the reference's ray cast (Body._test_if_targvec_visible,
 * body.py:2131-2150) instead of illumf's `visibl`. */
int pm_lonlat2xy_alt(const PMFrame *frame, const double *lon, const double *lat, int64_t n,
                     double alt, uint32_t flags, double *x, double *y, void *stream);

/*
 * Generic vectorised point transform between the coordinate systems above: replaces
 * SpiceBase._maybe_transform_as_arrays (base.py:718-757) driving the scalar pairs
 * BodyXY._xy2radec / _radec2xy / _xy2km / _km2xy / _xy2angular / _angular2xy (body_xy.py:409-676) and
 * Body._lonlat2radec / _radec2lonlat / _lonlat2angular / _angular2lonlat / _lonlat2km / _km2lonlat /
 * _radec2angular / _angular2radec / _radec2km / _km2radec / _km2angular / _angular2km
 * (body.py:1083-1900), plus graphic2centric_lonlat (LONLAT -> CENTRIC, body.py:2915-2947) and
 * centric2graphic_lonlat (LONLAT with PM_FLAG_PLANETOCENTRIC -> LONLAT, :2949-2982).
 *   a, b / out_a, out_b   first / second coordinate of every point (x, y | arcsec | km | RA, Dec deg |
 *                         lon, lat deg); non-finite inputs give NaN outputs
 *   alt                   LONLAT source: altitude of the point (pgrrec).  LONLAT destination: the frame must
 *                         carry the radii raised by alt (the reference's _AdjustedSurfaceAltitude); alt itself
 *                         is only used by the planetocentric output conversion
 *   flags                 PM_FLAG_NOT_VISIBLE_NAN (LONLAT source), PM_FLAG_PLANETOCENTRIC (LONLAT source: the
 *                         inputs are planetocentric; LONLAT destination: return planetocentric)
 *   aux13_host            HOST array: the 3 x 3 obsvec -> angular matrix of the ANGULAR system (row major;
 *                         Body._get_obsvec2angular_matrix for the caller's origin / rotation, body.py:1318-1343)
 *                         followed by the 2 x 2 km -> angular matrix (body.py:1625-1634); NULL = the frame's own
 *                         matrix and the inverse of its angular -> km matrix
 *   n_missed              device int64 (may be NULL): rays that missed the body on the way to lon / lat
 */
int pm_transform(const PMFrame *frame, int src, int dst, const double *a, const double *b, int64_t n,
                 double alt, uint32_t flags, const double *aux13_host, double *out_a, double *out_b,
                 int64_t *n_missed, void *stream);

/*
 * Time series: the three point transforms above for n_frames frames in ONE launch (what a fresh
 * BodyXY per epoch and one xy2lonlat / lonlat2xy / _transform call each do in the reference).
 * `frames`: n_frames (1 .. 65535) PMFrame structs in DEVICE memory, one per epoch, each packed as the
 * single-frame call of that epoch would use it (e.g. the altitude-adjusted frame for a lon / lat
 * destination with alt != 0).  Points: frame f reads a[f * point_stride + i], i < n; point_stride = 0
 * shares one set of n points between all frames, point_stride >= n gives every frame its own row.
 * Outputs: [n_frames][n].  n_missed: DEVICE int64[n_frames] (may be NULL), frame f's missed rays in
 * entry f.  aux13: DEVICE [n_frames][13], row f = pm_transform's aux13_host for frame f, or NULL for
 * every frame's defaults.  alt must be finite; flags as for the single-frame calls.
 * Row f of every output equals the single-frame call on frame f bit for bit.
 */
int pm_xy2lonlat_batch(const PMFrame *frames, int n_frames, const double *x, const double *y, int64_t n,
                       int64_t point_stride, double *lon, double *lat, int64_t *n_missed, void *stream);
int pm_lonlat2xy_batch(const PMFrame *frames, int n_frames, const double *lon, const double *lat, int64_t n,
                       int64_t point_stride, double alt, uint32_t flags, double *x, double *y, void *stream);
int pm_transform_batch(const PMFrame *frames, int n_frames, int src, int dst, const double *a, const double *b,
                       int64_t n, int64_t point_stride, double alt, uint32_t flags, const double *aux13,
                       double *out_a, double *out_b, int64_t *n_missed, void *stream);

/*
 * Inverse map projections, replacing pyproj.Transformer.transform(...,
 * direction='INVERSE') at body_xy.py:3126 for the three named non-rectangular
 * projections.  params = {a (r_eq), b (r_polar), lon_0, lat_0 (deg), lon_sign}.
 * xx, yy are in the projection's own units (body_xy.py:2905-2968 `to_meter`).
 * Output degrees; cells outside the projection are NaN.
 */
int pm_proj_inverse(int kind, const double *params5_host, const double *xx,
                    const double *yy, int64_t n, double *lon, double *lat, void *stream);
/* The forward direction of the same three projections (the default direction of the pyproj.Transformer
 * generate_map_coordinates returns, body_xy.py:3141-3153): planetographic lon / lat in degrees -> the
 * projection's own units; points the projection cannot show are NaN. */
int pm_proj_forward(int kind, const double *params5_host, const double *lon, const double *lat,
                    int64_t n, double *xx, double *yy, void *stream);

/*
 * Cube -> map resampling: replaces BodyXY._do_nearest_interpolation
 * (body_xy.py:1633-1649) and _do_spline_interpolation (:1651-1702) applied per
 * wavelength plane by Observation._get_mapped_data (observation.py:876-905).
 * Resamples planes [plane_begin, plane_begin + plane_count) of an n_planes cube:
 * xmap, ymap: [n_cells]; out: [plane_count][n_cells].  cells_per_row = length of a map row
 * when the cells form a regular 2-D grid (lets the dense-map cubic kernel work on 4 x 8
 * cell blocks that share one footprint), 0 if unknown; results do not depend on it.
 *   NEAREST:  `src` is the raw cube [n_planes][ny][nx]; nanbits / plane_bits unused.
 *   LINEAR / QUADRATIC / CUBIC: `src`, `nanbits`, `plane_bits` are the three buffers filled by
 *   pm_spline_prepare for the same (n_planes, ny, nx); plane_begin must be a multiple
 *   of 4.  Their layout is private to the library (plane-quad interleaved coefficients
 *   [ceil(n/4)][ny][nx][4], NaN bit planes [ny*nx][ceil(n/32)], per-word plane bits).
 */
int pm_gather(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits,
              int n_planes, int ny, int nx, int plane_begin, int plane_count,
              const double *xmap, const double *ymap, int64_t n_cells,
              int64_t cells_per_row, int mode, uint32_t flags, double *out, void *stream);

/*
 * NaN repair (BodyXY._replace_nans_with_interpolated_values, body_xy.py:1871-1904)
 * followed, for degree 2 / 3, by the separable interpolating B-spline fit scipy's
 * RectBivariateSpline(kx=ky=degree, s=0) performs (body_xy.py:1673-1680; FITPACK knots:
 * not-a-knot for degree 3, mid-sample knots for degree 2), packed for
 * pm_gather.  In: cube [n_planes][ny][nx].  Out: coef (pm_spline_coef_bytes),
 * nanbits (pm_spline_nanbits_bytes), plane_bits (pm_spline_planebits_bytes).
 * `work` must hold pm_spline_work_bytes(...) bytes of device scratch.
 */
int64_t pm_spline_coef_bytes(int n_planes, int ny, int nx);
int64_t pm_spline_nanbits_bytes(int n_planes, int ny, int nx);
int64_t pm_spline_planebits_bytes(int n_planes);
int64_t pm_spline_work_bytes(int n_planes, int ny, int nx, int degree);
int pm_spline_prepare(const double *cube, int n_planes, int ny, int nx, int degree,
                      double *coef, uint32_t *nanbits, uint32_t *plane_bits, void *work,
                      void *stream);

/*
 * Smoothing splines, map_img(spline_smoothing = s > 0): per plane, FITPACK's regrid (iopt 0, maxit as
 * given, tol 0.001, nxest = ny + k_rows + 1, nyest = nx + k_cols + 1), i.e. RectBivariateSpline(
 * arange(ny), arange(nx), plane, kx = k_rows, ky = k_cols, s) (body_xy.py:1651-1702), one CTA per plane
 * and one launch for any number of planes.  `coef` / `plane_bits` are pm_spline_prepare's outputs for
 * degree PM_INTERP_LINEAR (the NaN-repaired planes); all-NaN planes are not fitted (nx = ny = 0,
 * ier 0, fp NaN).  Per plane l, in fixed-size slots:
 *   tx [n_planes][ny + k_rows + 1], ty [n_planes][nx + k_cols + 1], c [n_planes][ny * nx]
 *   (c[l][i * (ny_l - k_cols - 1) + j] multiplies B_i(row) B_j(column)), nxy [n_planes][2] = knot
 *   counts (nx_l along rows, ny_l along columns), fp [n_planes], ier [n_planes] = FITPACK's ier
 *   (0, -1, -2 accepted by RectBivariateSpline; 1, 2, 3 are its ValueErrors).
 * `work` must hold pm_regrid_work_bytes(...) bytes of device scratch.  k_rows, k_cols: 1..3.
 */
int64_t pm_regrid_work_bytes(int n_planes, int ny, int nx, int k_rows, int k_cols);
int pm_regrid_fit(const double *coef, const uint32_t *plane_bits, int n_planes, int ny, int nx, int k_rows,
                  int k_cols, double s, int maxit, double *tx, double *ty, double *c, int *nxy, double *fp,
                  int *ier, void *work, void *stream);
/*
 * Evaluation of pm_regrid_fit's splines at map cells (RectBivariateSpline.ev(y, x), bispeu): planes
 * [plane_begin, plane_begin + plane_count), any plane_begin; out [plane_count][n_cells].  NaN cells,
 * all-NaN planes and (flags PM_FLAG_PROPAGATE_NAN) the cells of _should_propagate_nan_to_map are NaN,
 * as in pm_gather; nanbits / plane_bits are pm_spline_prepare's.
 */
int pm_gather_regrid(const double *tx, const double *ty, const double *c, const int *nxy,
                     const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes, int ny, int nx,
                     int k_rows, int k_cols, int plane_begin, int plane_count, const double *xmap,
                     const double *ymap, int64_t n_cells, uint32_t flags, double *out, void *stream);

/*
 * map_img(interpolation='smooth') (BodyXY._do_smooth_interpolation, body_xy.py:1704-1790):
 *   pm_nan_minmax         np.nanmin / np.nanmax of a device array -> out2[2] (device), the x / y
 *                         map limits the host needs to size the oversampled grid (:1720-1721);
 *   pm_pchip_resample     BodyXY._pchip_grid_interp2d (:1792-1853): PchipInterpolator over the
 *                         finite pixels of columns x_first..x_last of every row y_first..y_last,
 *                         then of every column, evaluated on np.linspace(first, last, n) grids;
 *                         fine: [n_planes][n_ys][n_xs]; `work`: pm_pchip_work_bytes(...) bytes;
 *   pm_gather_grid_linear RegularGridInterpolator(method='linear', bounds_error=False,
 *                         fill_value=nan) on `fine` at (ymap, xmap) with the propagate_nan rule
 *                         evaluated on the original cube (:1761-1790); out: [n_planes][n_cells].
 */
int pm_nan_minmax(const double *x, int64_t n, double *out2, void *stream);
int64_t pm_pchip_work_bytes(int n_planes, int ny, int nx, int n_xs);
int pm_pchip_resample(const double *cube, int n_planes, int ny, int nx, int x_first, int x_last,
                      int y_first, int y_last, int n_xs, int n_ys, double *fine, void *work,
                      void *stream);
int pm_gather_grid_linear(const double *fine, int n_planes, int n_ys, int n_xs, int x_first,
                          int x_last, int y_first, int y_last, const double *cube, int ny, int nx,
                          const double *xmap, const double *ymap, int64_t n_cells, uint32_t flags,
                          double *out, void *stream);

/* FP64 FMA throughput probe used by bench.py for the compute roofline
 * denominator: runs `iters` dependent-chain DFMAs per thread on a full grid and
 * returns the kernel time in ms through *ms_host (synchronises). */
int pm_fp64_peak_probe(int iters, double *ms_host, double *flops_host);
/* The same probe for two operand mixes: kind 0 = one register operand per DFMA (pm_fp64_peak_probe, the
 * datasheet rate), kind 1 = three distinct register operands per DFMA, the form per-pixel vector algebra
 * issues; the register file feeds that form at 2/3 of the rate (measured: profiles/r2_summary.md). */
int pm_fp64_probe(int kind, int iters, double *ms_host, double *flops_host);

/*
 * FITS staging for Observation.save_observation (observation.py:1185-1303) and
 * save_mapped_observation (:1315-1474).  Both append one `fits.ImageHDU(data=float64 array)`
 * per backplane (EXTNAME = backplane name, :1281-1284 / :1434-1441) after the primary HDU and
 * let astropy (third party, astropy.io.fits) write them: each data unit is the array as
 * big-endian IEEE-754 doubles zero-padded to a multiple of 2880 bytes.
 * pm_fits_stage converts n_units device arrays into their data units inside ONE
 * device-resident image of the file, so the file leaves the device in a single copy:
 *   src[u]         device pointer to the n_elems[u] doubles of unit u (native byte order)
 *   dst_offset[u]  byte offset of unit u's data unit inside `image` (a multiple of 8; FITS
 *                  layouts make it a multiple of 2880)
 *   image          device buffer holding the file; header blocks are the caller's (host-built)
 * src, n_elems and dst_offset are HOST arrays of n_units entries (read before returning).
 * pm_fits_data_unit_bytes(n) = the padded size of an n-element float64 data unit.
 */
#define PM_FITS_MAX_UNITS 32 /* units per launch; more are split over several launches */
int64_t pm_fits_data_unit_bytes(int64_t n_elems);
int pm_fits_stage(const double *const *src, const int64_t *n_elems, const int64_t *dst_offset,
                  int n_units, uint8_t *image, void *stream);

/*
 * HOST functions (no device work): the two ephemeris primitives behind the once-per-frame
 * constants when spiceypy is not the provider.  They replace, for SPK types 2 / 3 and the text-PCK
 * IAU orientation model, the CSPICE calls the reference makes through spiceypy: spkssb / spkezr
 * (planetmapper/base.py:828) and the pxform / sxform rotations (body.py:935-945, base.py:815-837).
 *   pm_host_ssb_state    state (km, km/s) of `body` relative to the solar-system barycentre, J2000,
 *                        summed along the centre chain; `segs` in precedence order (the last
 *                        loaded kernel first), `records` the concatenated Chebyshev records.
 *                        PM_ERR_UNSUPPORTED: no segment covers (body, et).
 *   pm_host_orientation  J2000 -> body-fixed rotation R (row major, v_body = R v_j2000) at et and the
 *                        angular velocity omega of the body frame in body axes (dR/dt = -[omega]x R).
 */
#define PM_MAX_NUT_TERMS 64
typedef struct PMEphemSegment {
    int32_t target, center, spk_type, rsize; /* NAIF ids, SPK type 2 or 3, doubles per record        */
    int32_t n, first_record, n_kept, pad;    /* records in the segment; kept slice [first, first + kept) */
    double et_start, et_end, init, intlen;   /* coverage; first record start and record length (s)   */
    int64_t rec_offset;                      /* index of the first kept record in `records` (doubles) */
} PMEphemSegment;
typedef struct PMOrientationModel {
    double pole_ra[3], pole_dec[3], pm[3];   /* BODYnnn_POLE_RA / POLE_DEC / PM (deg, deg/century or /day) */
    int32_t n_ra, n_dec, n_pm, n_nut;        /* polynomial lengths; number of NUT_PREC_ANGLES pairs   */
    int32_t n_nut_ra, n_nut_dec, n_nut_pm, pad;
    double nut_ra[PM_MAX_NUT_TERMS], nut_dec[PM_MAX_NUT_TERMS], nut_pm[PM_MAX_NUT_TERMS];
    double nut_angles[2 * PM_MAX_NUT_TERMS]; /* (deg, deg/century) pairs of the system barycentre     */
} PMOrientationModel;
int pm_host_ssb_state(const PMEphemSegment *segs, int n_segs, const double *records, int body,
                      double et, double *state6);
int pm_host_orientation(const PMOrientationModel *model, double et, double *rmat9, double *omega3);

/* Diagnostic: evaluates one of the library's own FP64 primitives (the MUFU-seeded
 * reciprocal / rsqrt / sqrt / division and the polynomial sin / cos / atan2 / acos
 * that replace CUDA's libm on the hot path) elementwise, so tests can measure their
 * ulp error on the device.  kind: 0 rcp(a), 1 rsqrt(a), 2 sqrt(a), 3 sin(a) and
 * 4 cos(a) for |a| <= pi/4, 5 atan2(a, b), 6 acos(a), 7 a / b, 8 sin(a), 9 cos(a)
 * for any |a| < 1e5, 10 atan2(|a|, b) and 11 atan2(a, |b|) (the half-plane variants used
 * for vector separations and latitudes), 12 sin(a) and 13 cos(a) as the pixel-offset path
 * evaluates them (a tiny-angle series for |a| <= 2^-8, else as 3 / 4).  `b` may be NULL for the
 * one-argument kinds. */
int pm_math_probe(int kind, const double *a, const double *b, int64_t n, double *out,
                  void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PM_B200_H */
