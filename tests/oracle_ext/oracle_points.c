/*
 * oracle_points.c - TEST INFRASTRUCTURE ONLY.
 *
 * Two references for the per-point geometry queries, built on the CPU oracle's own routines:
 * the oracle source is compiled into this translation unit unchanged (so its static helpers are
 * reachable) and the two entries below only loop over them.  Built by tests/test_points_host.py
 * into a temporary directory with the oracle's flags (oracle/Makefile: -ffp-contract=off).
 *
 *   pmox_backplanes_points  the oracle's per-pixel code (pixel_backplanes) at n arbitrary FINITE image
 *                           positions, fractional or outside the image; out: [popcount(mask)][n],
 *                           margin as pmo_backplanes_img
 *   pmox_ring_coordinates   Body.ring_plane_coordinates(ra, dec, only_visible=False) (body.py:2577-2615):
 *                           the ring-plane point along each RA / Dec direction (degrees), not hidden by
 *                           the body
 */
#include "../../oracle/pm_oracle.c"

int pmox_backplanes_points(const PMFrame *f, const double *x, const double *y, int64_t n, uint64_t mask,
                           double *out, double *margin) {
    if (!f || n < 0) return PM_ERR_BAD_ARG;
    if (n > 0 && (!x || !y || !out)) return PM_ERR_BAD_ARG;
    mask &= PM_ALL_PLANES;
    for (int64_t i = 0; i < n; i++) {
        PixelOut o;
        pixel_backplanes(f, x[i], y[i], mask, &o);
        int slot = 0;
        for (int k = 0; k < PM_N_PLANES; k++) {
            if (mask & (1ull << k)) {
                out[(int64_t)slot * n + i] = o.v[k];
                slot++;
            }
        }
        if (margin) margin[i] = o.margin;
    }
    return PM_OK;
}

int pmox_ring_coordinates(const PMFrame *f, const double *ra, const double *dec, int64_t n, double *radius,
                          double *lon, double *dist) {
    if (!f || n < 0) return PM_ERR_BAD_ARG;
    if (n > 0 && (!ra || !dec || !radius || !lon || !dist)) return PM_ERR_BAD_ARG;
    for (int64_t i = 0; i < n; i++) {
        double d[3];
        radec_deg2obsvec_norm(ra[i], dec[i], d);
        ring_coordinates(f, d, &radius[i], &lon[i], &dist[i]);
    }
    return PM_OK;
}
