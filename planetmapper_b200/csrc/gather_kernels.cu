// gather_kernels.cu - cube -> map resampling (nearest / linear / not-a-knot cubic)
// and the spline preparation (NaN repair + B-spline coefficient solve).
//
// Replaces, for every wavelength plane at once, BodyXY._do_nearest_interpolation
// (planetmapper/body_xy.py:1633-1649), BodyXY._do_spline_interpolation
// (:1651-1702, scipy RectBivariateSpline s=0 -> FITPACK), _should_propagate_nan_to_map
// (:1855-1866) and _replace_nans_with_interpolated_values (:1871-1904), which
// Observation._get_mapped_data (planetmapper/observation.py:876-905) runs plane by
// plane in Python.
//
// Gather layout: thread = map cell (consecutive threads -> consecutive cells, so each
// plane's store is one coalesced 256 B warp transaction, written with a streaming
// hint because the output is never re-read); the per-cell interpolation weights are
// computed ONCE and reused for every wavelength plane of the CTA's plane group.
// The kernel is HBM-write bound: 8 B per output voxel.
#include "pm_device.cuh"
#include "pm_kernels.h"

#include <type_traits>

#include <cstdlib>
#include <map>
#include <utility>
#include <mutex>
#include <vector>

namespace pm {

constexpr int kGatherBlock = 256;
constexpr uint8_t kPlaneAllNan = 1;  // plane_skip bit0: np.all(np.isnan(img)) -> all NaN out
constexpr uint8_t kPlaneHasNan = 2;  // plane_skip bit1: some NaN pixel -> consult nanmask

// FITPACK's interpolating-spline knot vectors (s = 0) for n samples at 0..n-1:
//   degree 3 (not-a-knot):  t = [0,0,0,0, 2,3,...,n-3, n-1,n-1,n-1,n-1]
//   degree 2 (knots between the samples): t = [0,0,0, 1.5,2.5,...,n-2.5, n-1,n-1,n-1]
template <int DEG>
__host__ __device__ __forceinline__ double spline_knot(int i, int n) {
    if (i <= DEG) return 0.0;
    if (i >= n) return (double)(n - 1);
    return DEG == 3 ? (double)(i - 2) : (double)i - 1.5;
}

// FITPACK fpbspl: the DEG + 1 non-zero B-splines at x; returns the first coefficient
// index.  x is clamped to [0, n-1] like bispev does.
template <int DEG>
__host__ __device__ __forceinline__ int bspline_weights(double x, int n, double h[DEG + 1]) {
    double xe = fmin(fmax(x, 0.0), (double)(n - 1));
    int l = (DEG == 3) ? (int)floor(xe) + 2 : (int)floor(xe + 1.5);
    l = l < DEG ? DEG : (l > n - 1 ? n - 1 : l);
    double hh[DEG];
    h[0] = 1.0;
#pragma unroll
    for (int i = 1; i <= DEG; i++) h[i] = 0.0;
#pragma unroll
    for (int jj = 1; jj <= DEG; jj++) {
#pragma unroll
        for (int i = 0; i < DEG; i++)
            if (i < jj) hh[i] = h[i];
        h[0] = 0.0;
#pragma unroll
        for (int i = 0; i < DEG; i++) {
            if (i < jj) {
                int li = l + 1 + i, lj = li - jj;
                double tli = spline_knot<DEG>(li, n), tlj = spline_knot<DEG>(lj, n);
                double f = fast_div(hh[i], tli - tlj);  // knot spans are small half-integers: exact or correctly rounded
                h[i] = h[i] + f * (tli - xe);
                h[i + 1] = f * (xe - tlj);
            }
        }
    }
    return l - DEG;
}
__host__ __device__ __forceinline__ int bspline3_weights(double x, int n, double h[4]) {
    return bspline_weights<3>(x, n, h);
}

// ---------------------------------------------------------------------------------
// nearest neighbour: reads the raw cube [n_planes][ny][nx]
// ---------------------------------------------------------------------------------
// Planes plane_begin + [l0, l1) at map cell `cell` into out[l][cell]
__device__ __forceinline__ void nearest_cell_planes(const double *__restrict__ cube, int ny, int nx, int plane_begin,
                                                    int l0, int l1, const double *__restrict__ xmap,
                                                    const double *__restrict__ ymap, int64_t cell, int64_t n_cells,
                                                    double *__restrict__ out) {
    const int64_t plane_px = (int64_t)ny * nx;
    const double x = __ldg(xmap + cell), y = __ldg(ymap + cell);
    const double nan = NAN;
    bool valid = !isnan(x);  // y is never NaN when x is not (body_xy.py:1646, :1697)
    int64_t off = 0;
    if (valid) {
        // np.round is round-half-to-even == rint (body_xy.py:1642-1643)
        long xi = (long)rint(x), yi = isnan(y) ? -999 : (long)rint(y);
        if (xi < 0) xi += nx;  // numpy negative indices wrap
        if (yi < 0) yi += ny;
        valid = xi >= 0 && xi < nx && yi >= 0 && yi < ny;
        off = (int64_t)yi * nx + xi;
    }
    const double *src = cube + (int64_t)(plane_begin + l0) * plane_px + off;
    double *dst = out + (int64_t)l0 * n_cells + cell;
    int l = l0;
    for (; l + 4 <= l1; l += 4) {
        double v0 = nan, v1 = nan, v2 = nan, v3 = nan;
        if (valid) {
            v0 = __ldg(src);
            v1 = __ldg(src + plane_px);
            v2 = __ldg(src + 2 * plane_px);
            v3 = __ldg(src + 3 * plane_px);
        }
        __stcs(dst, v0);
        __stcs(dst + n_cells, v1);
        __stcs(dst + 2 * n_cells, v2);
        __stcs(dst + 3 * n_cells, v3);
        src += 4 * plane_px;
        dst += 4 * n_cells;
    }
    for (; l < l1; l++) {
        __stcs(dst, valid ? __ldg(src) : nan);
        src += plane_px;
        dst += n_cells;
    }
}
__global__ void __launch_bounds__(kGatherBlock)
    gather_nearest_kernel(const double *__restrict__ cube, int ny, int nx, int plane_begin, int plane_count,
                          const double *__restrict__ xmap, const double *__restrict__ ymap, int64_t n_cells,
                          double *__restrict__ out, int planes_per_group) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= n_cells) return;
    const int l0 = blockIdx.y * planes_per_group;
    const int l1 = min(l0 + planes_per_group, plane_count);
    nearest_cell_planes(cube, ny, nx, plane_begin, l0, l1, xmap, ymap, cell, n_cells, out);
}

// ---------------------------------------------------------------------------------
// spline modes: read the prepared operand of pm_spline_prepare
//   coefq   [ceil(n_planes / 4)][ny][nx][4]   four wavelength planes of one pixel are
//           32 contiguous bytes, so one 256-bit load feeds four FMAs and the K x K
//           footprint of a cell is K runs of K x 32 contiguous bytes;
//   nanbits [ny * nx][n_words]                bit (l % 32) of word l / 32 = pixel was NaN
//           in plane l: the propagate_nan test costs four word loads per 32 planes;
//   plane_bits [2][n_words]                   row 0: all-NaN planes, row 1: words with any
//           NaN pixel (nanbits needs consulting).
// The K x K weight products are formed once per cell; per output voxel the kernel then
// issues K*K/4 loads, K*K FMAs and one streaming store.
// ---------------------------------------------------------------------------------
struct Quad {
    double v[4];
};
__device__ __forceinline__ Quad ldg_quad(const double *p) {
    Quad q;
    asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(q.v[0]), "=d"(q.v[1]), "=d"(q.v[2]), "=d"(q.v[3])
                 : "l"(p));
    return q;
}

// The K = degree + 1 non-zero basis functions of one axis at coordinate x (n samples);
// returns the first coefficient index.  K = 2 is the degree-1 spline = linear interpolation
// with bispev's clamping.
template <int K>
__device__ __forceinline__ int axis_weights(double x, int n, double w[K]) {
    if (K == 2) {
        const double xe = fmin(fmax(x, 0.0), (double)(n - 1));
        const int i = min((int)floor(xe), n - 2);
        const double fx = xe - i;
        w[0] = 1.0 - fx;
        w[1] = fx;
        return i;
    }
    return bspline_weights<(K == 2 ? 2 : K - 1)>(x, n, w);
}

// Per-cell state of the spline gather (weights, footprint origin, NaN-test pixels)
template <int KY, int KX>
struct CellState {
    double w[KY * KX];   // wy[a] * wx[b], FITPACK fpbisp order (rows outer)
    int64_t origin;      // ((iy * nx + ix) * 4): offset of the footprint inside a plane quad
    uint32_t nb[4];      // pixel indices floor/ceil(x, y) for _should_propagate_nan_to_map
    uint32_t bad;        // NaN bits of the current 32-plane word
    bool valid;
};
template <int KY, int KX>
__device__ __forceinline__ void setup_cell(CellState<KY, KX> &c, double x, double y, int ny, int nx,
                                           bool propagate) {
    c.valid = !isnan(x);  // y is never NaN when x is not (body_xy.py:1646, :1697)
    c.bad = 0;
    c.origin = 0;
    c.nb[0] = c.nb[1] = c.nb[2] = c.nb[3] = 0;
    if (c.valid && propagate) {
        // BodyXY._should_propagate_nan_to_map (body_xy.py:1855-1866)
        if (x < 0.0 || y < 0.0 || x > nx - 1 || y > ny - 1) c.valid = false;
        const int x0 = max((int)floor(x), 0), x1 = min((int)ceil(x), nx - 1);
        const int y0 = max((int)floor(y), 0), y1 = min((int)ceil(y), ny - 1);
        c.nb[0] = (uint32_t)(y0 * nx + x0);
        c.nb[1] = (uint32_t)(y0 * nx + x1);
        c.nb[2] = (uint32_t)(y1 * nx + x0);
        c.nb[3] = (uint32_t)(y1 * nx + x1);
    }
    if (c.valid) {
        double wx[KX], wy[KY];
        const int ix = axis_weights<KX>(x, nx, wx);
        const int iy = axis_weights<KY>(y, ny, wy);
#pragma unroll
        for (int a = 0; a < KY; a++)
#pragma unroll
            for (int b = 0; b < KX; b++) c.w[a * KX + b] = wy[a] * wx[b];
        c.origin = ((int64_t)iy * nx + ix) * 4;
    } else {
#pragma unroll
        for (int k = 0; k < KY * KX; k++) c.w[k] = 0.0;
    }
}

// Planes plane_begin + [l0, l1) of one prepared cell, a plane quad at a time (plane_begin + l0 a multiple
// of 4), into out[l][cell]
template <int KY, int KX>
__device__ __forceinline__ void spline_cell_quads(CellState<KY, KX> &cs, const double *__restrict__ coefq,
                                                  const uint32_t *__restrict__ nanbits,
                                                  const uint32_t *__restrict__ plane_bits, int n_words, int ny,
                                                  int nx, int plane_begin, int l0, int l1, bool propagate,
                                                  int64_t cell, int64_t n_cells, double *__restrict__ out) {
    const double nan = NAN;
    const int64_t quad_stride = (int64_t)ny * nx * 4;  // doubles per plane quad
    const int64_t row_stride = (int64_t)nx * 4;
    const double *src = coefq + (int64_t)((plane_begin + l0) >> 2) * quad_stride + cs.origin;
    double *dst = out + (int64_t)l0 * n_cells + cell;
    int cur_word = -1;
    for (int l = l0; l < l1; l += 4) {
        const int gl = plane_begin + l;  // global plane index of this quad (multiple of 4)
        const int word = gl >> 5;
        if (word != cur_word) {  // uniform: once per 32 planes
            cur_word = word;
            uint32_t bad = __ldg(plane_bits + word);
            if (cs.valid && propagate && __ldg(plane_bits + n_words + word)) {
#pragma unroll
                for (int k = 0; k < 4; k++) bad |= __ldg(nanbits + (int64_t)cs.nb[k] * n_words + word);
            }
            cs.bad = bad;
        }
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        if (cs.valid) {
#pragma unroll
            for (int a = 0; a < KY; a++) {
#pragma unroll
                for (int b = 0; b < KX; b++) {
                    const Quad q = ldg_quad(src + a * row_stride + b * 4);
                    const double ww = cs.w[a * KX + b];
#pragma unroll
                    for (int j = 0; j < 4; j++) acc[j] = fma(q.v[j], ww, acc[j]);
                }
            }
        }
        const uint32_t nib = cs.valid ? ((cs.bad >> (gl & 31)) & 0xFu) : 0xFu;
        const int left = l1 - l;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j < left) __stcs(dst + (int64_t)j * n_cells, ((nib >> j) & 1u) ? nan : acc[j]);
        }
        src += quad_stride;
        dst += 4 * n_cells;
    }
}

// Plane gl (any index) of one prepared cell, read from its lane of the plane quad: per plane the same loads,
// FMAs (rows outer) and NaN words as spline_cell_quads, so the two agree bit for bit
template <int KY, int KX>
__device__ __forceinline__ double spline_cell_plane(const CellState<KY, KX> &cs, const double *__restrict__ coefq,
                                                    const uint32_t *__restrict__ nanbits,
                                                    const uint32_t *__restrict__ plane_bits, int n_words, int ny,
                                                    int nx, int gl, bool propagate) {
    if (!cs.valid) return NAN;
    const int word = gl >> 5;
    uint32_t bad = __ldg(plane_bits + word);
    if (propagate && __ldg(plane_bits + n_words + word)) {
#pragma unroll
        for (int k = 0; k < 4; k++) bad |= __ldg(nanbits + (int64_t)cs.nb[k] * n_words + word);
    }
    if ((bad >> (gl & 31)) & 1u) return NAN;
    const int64_t row_stride = (int64_t)nx * 4;
    const double *p = coefq + (int64_t)(gl >> 2) * ny * row_stride + cs.origin + (gl & 3);
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < KY; a++)
#pragma unroll
        for (int b = 0; b < KX; b++) acc = fma(__ldg(p + a * row_stride + b * 4), cs.w[a * KX + b], acc);
    return acc;
}

// One cell per thread, KY x KX footprint (KY = row degree + 1, KX = column degree + 1)
template <int KY, int KX, int kMinBlocks>
__global__ void __launch_bounds__(kGatherBlock, kMinBlocks)
    gather_spline_kernel(const double *__restrict__ coefq, const uint32_t *__restrict__ nanbits,
                         const uint32_t *__restrict__ plane_bits, int n_words, int ny, int nx, int plane_begin,
                         int plane_count, const double *__restrict__ xmap, const double *__restrict__ ymap,
                         int64_t n_cells, uint32_t flags, double *__restrict__ out, int planes_per_group) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= n_cells) return;
    const int l0 = blockIdx.y * planes_per_group;  // relative to plane_begin, multiple of 4
    const int l1 = min(l0 + planes_per_group, plane_count);
    const bool propagate = (flags & PM_FLAG_PROPAGATE_NAN) != 0;
    CellState<KY, KX> cs;
    setup_cell<KY, KX>(cs, __ldg(xmap + cell), __ldg(ymap + cell), ny, nx, propagate);
    spline_cell_quads<KY, KX>(cs, coefq, nanbits, plane_bits, n_words, ny, nx, plane_begin, l0, l1, propagate, cell,
                              n_cells, out);
}

// ---------------------------------------------------------------------------------
// Cubic gather for maps much finer than the image (the C4 case: ~1500 cells per pixel).
//
// For cells that share a 4 x 4 footprint the interpolation is a small dense product
//     out[plane][cell] = sum_k coef[plane][k] * w[k][cell],   k = 0..15,
// and the one-cell-per-thread kernel above is bound by the L1 -> register return path
// (every voxel pulls its 16 coefficients = 128 B through a 128 B/clk/SM pipe: ncu shows
// l1tex__data_pipe_lsu_wavefronts at 82 % while DRAM sits at 45 %).  Sharing loaded
// coefficients between the cells of one thread (C = 2) only moves the bound to register
// pressure.  The warp-level FP64 MMA (DMMA.8x8x4) is the register-tiled form of exactly
// this product: a warp owns 32 consecutive cells and streams planes 8 at a time,
//     A (8 planes x 4 coefficients)  one coefficient per lane, loaded once per footprint,
//     B (4 coefficients x 8 cells)   the cell weights, held in registers for all planes,
//     D (8 planes x 8 cells)         two voxels per lane,
// so a voxel costs 16 B of L1 traffic instead of 128 B.  Cells of an 8-cell tile that do
// NOT share the footprint are handled by repeating the product per distinct footprint
// with the other cells' weights zeroed, so the result is exact for any map; the launcher
// only selects this kernel when the map is dense enough for sharing to be the rule.
// The arithmetic is IEEE FP64 FMA like the scalar kernel (accumulation order differs).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void dmma8x8x4(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// The A fragments are staged through shared memory with cp.async: one 8-byte copy per lane and
// coefficient row, each lane reading back exactly what it copied (no cross-lane exchange, no
// barrier).  What this buys is the GROUP accounting: `cp.async.wait_group N` waits for the
// oldest group only, so the next plane tile is genuinely in flight while one is multiplied.  The earlier
// register-prefetch version compiled to loads that all shared one hardware scoreboard (SASS:
// every LDG of the three rotating register sets wrote SB5); waiting for the tile about to be
// multiplied therefore also waited for the prefetches just issued.
constexpr int kCubicBlock = 128;   // threads per CTA: 4 CTAs / SM at <= 128 registers, fine-grained tail
#ifndef PM_CUBIC_SLOTS
#define PM_CUBIC_SLOTS 6
#endif
constexpr int kCubicSlots = PM_CUBIC_SLOTS;  // 1 KB footprint slots per warp: 6 = 24 KB per CTA, 96 KB per SM at four CTAs

__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gsrc) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(double *smem_dst, const double *gsrc) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
#ifdef PM_CUBIC_CG
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");   // L2 only
#else
    // through L1: ~47 warps per image pixel re-read the same coefficient quads
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

#ifndef PM_CUBIC_CTAS
#define PM_CUBIC_CTAS 4
#endif
__global__ void __launch_bounds__(kCubicBlock, PM_CUBIC_CTAS)
    gather_cubic_mma_kernel(const double *__restrict__ coefq, const uint32_t *__restrict__ nanbits,
                            const uint32_t *__restrict__ plane_bits, int n_words, int ny, int nx, int n_planes_padded,
                            int plane_begin, int plane_count, const double *__restrict__ xmap,
                            const double *__restrict__ ymap, int64_t n_cells, int64_t row_len, uint32_t flags,
                            double *__restrict__ out, int planes_per_group, int lead) {
    // plane_begin is a multiple of 8 here: a plane tile (8 planes) then never straddles a 32-plane NaN word,
    // which keeps refresh_ok's warp shuffles uniform.  A caller's range starting on an odd quad is launched
    // from the quad before it with lead = 4: the first `lead` planes are computed but not stored, and `out`
    // already points `lead` planes before the caller's buffer.
    constexpr unsigned kFull = 0xffffffffu;
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    // Warp -> cells.  With a known map row length (row_len < n_cells) a warp owns a block of
    // 4 map rows x 8 columns (tile i = row i of the block): neighbouring rows and columns
    // almost always share one 4 x 4 footprint.  Otherwise it owns 32 consecutive cells
    // (tile i = cells 8 i .. 8 i + 7).
    const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const bool grid2d = row_len < n_cells;
    int64_t base0, tile_step;
    int ncols[4];
    if (grid2d) {
        const int64_t col_tiles = (row_len + 7) / 8, n_rows = n_cells / row_len;
        const int64_t rg = warp_id / col_tiles, ct = warp_id - rg * col_tiles;
        if (4 * rg >= n_rows) return;  // whole warp
        base0 = 4 * rg * row_len + 8 * ct;
        tile_step = row_len;
        const int nc = (int)min((int64_t)8, row_len - 8 * ct);
#pragma unroll
        for (int i = 0; i < 4; i++) ncols[i] = (4 * rg + i < n_rows) ? nc : 0;
    } else {
        base0 = 32 * warp_id;
        if (base0 >= n_cells) return;  // whole warp
        tile_step = 8;
#pragma unroll
        for (int i = 0; i < 4; i++) ncols[i] = (int)max((int64_t)0, min((int64_t)8, n_cells - base0 - 8 * i));
    }
    const int l0 = blockIdx.y * planes_per_group;  // relative to plane_begin, multiple of 8
    const int l1 = min(l0 + planes_per_group, plane_count);
    const double nan = NAN;
    const bool propagate = (flags & PM_FLAG_PROPAGATE_NAN) != 0;

    // ---- per-cell setup.  Lane L works out cell (tile L >> 3, column L & 7) ONCE - map load, validity,
    // NaN-test pixels, B-spline weights (the not-a-knot weights are ~250 instructions per axis) -
    // then the values travel to the four lanes (g, t = 0..3) that describe that cell in the MMA.
    double bw[4][4];          // B fragments: bw[i][j] = wy[j] * wx[t] of tile i's cell g
    uint32_t origin[4];       // iy * nx + ix of the footprint (pixel index)
    uint32_t nbp[4];          // NaN-test pixels, packed: x0 | y0 << 14 | (x1 - x0) << 28 | (y1 - y0) << 29
    uint32_t cls[4];          // lanes of the tile sharing this lane's footprint
    uint32_t valid_mask[4];   // ballot of valid cells per tile
    {
        const int ti = lane >> 3, col = lane & 7;
        const int nc = ti == 0 ? ncols[0] : (ti == 1 ? ncols[1] : (ti == 2 ? ncols[2] : ncols[3]));
        const int64_t cell = base0 + ti * tile_step + col;
        const bool in_range = col < nc;
        const double x = in_range ? __ldg(xmap + cell) : nan, y = in_range ? __ldg(ymap + cell) : nan;
        bool valid = !isnan(x);  // y is never NaN when x is not (body_xy.py:1646, :1697)
        uint32_t my_nbp = 0, my_origin = 0xffffffffu;
        if (valid && propagate) {
            // BodyXY._should_propagate_nan_to_map (body_xy.py:1855-1866)
            if (x < 0.0 || y < 0.0 || x > nx - 1 || y > ny - 1) valid = false;
            const int x0 = max((int)floor(x), 0), x1 = min((int)ceil(x), nx - 1);
            const int y0 = max((int)floor(y), 0), y1 = min((int)ceil(y), ny - 1);
            my_nbp = (uint32_t)x0 | ((uint32_t)y0 << 14) | ((uint32_t)(x1 > x0) << 28) | ((uint32_t)(y1 > y0) << 29);
        }
        double wx[4] = {0.0, 0.0, 0.0, 0.0}, wy[4] = {0.0, 0.0, 0.0, 0.0};
        if (valid) {
            const int ix = bspline3_weights(x, nx, wx);
            const int iy = bspline3_weights(y, ny, wy);
            my_origin = (uint32_t)(iy * nx + ix);
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int src = 8 * i + g;  // the lane that worked out cell g of tile i
            origin[i] = __shfl_sync(kFull, my_origin, src);
            nbp[i] = __shfl_sync(kFull, my_nbp, src);
            valid_mask[i] = __ballot_sync(kFull, origin[i] != 0xffffffffu);
            const double w0 = __shfl_sync(kFull, wx[0], src), w1 = __shfl_sync(kFull, wx[1], src);
            const double w2 = __shfl_sync(kFull, wx[2], src), w3 = __shfl_sync(kFull, wx[3], src);
            const double wxt = t == 0 ? w0 : (t == 1 ? w1 : (t == 2 ? w2 : w3));
#pragma unroll
            for (int j = 0; j < 4; j++) bw[i][j] = __shfl_sync(kFull, wy[j], src) * wxt;  // zero for invalid cells
            cls[i] = __match_any_sync(kFull, origin[i]);
        }
    }
    if ((valid_mask[0] | valid_mask[1] | valid_mask[2] | valid_mask[3]) == 0) {
        // nothing visible in these 32 cells: stream NaN; 16 lanes x 16 B cover one plane
        const int ti = (lane & 15) >> 2, pr = lane & 3;
        const int nc = ti == 0 ? ncols[0] : (ti == 1 ? ncols[1] : (ti == 2 ? ncols[2] : ncols[3]));
        const int64_t cell = base0 + ti * tile_step + 2 * pr;
        const bool aligned = ((n_cells & 1) == 0) && (!grid2d || (row_len & 1) == 0);
        const int skip = l0 < lead ? lead - l0 : 0;  // (even) planes of the first tile that belong to the quad before
        double *d = out + (int64_t)(l0 + skip + (lane >> 4)) * n_cells + cell;
        const int64_t step2 = 2 * n_cells;
        const int n_it = (l1 - l0 - skip - (lane >> 4) + 1) / 2;  // planes l0 + skip + (lane >> 4), + 2, ... < l1
        if (aligned && 2 * pr + 1 < nc) {
#pragma unroll 4
            for (int it = 0; it < n_it; it++, d += step2)
                asm volatile("st.global.cs.v2.f64 [%0], {%1, %1};" ::"l"(d), "d"(nan) : "memory");
        } else {
            for (int it = 0; it < n_it; it++, d += step2) {
                if (2 * pr < nc) __stcs(d, nan);
                if (2 * pr + 1 < nc) __stcs(d + 1, nan);
            }
        }
        return;
    }

    const int64_t quad_stride = (int64_t)ny * nx * 4;
    const int64_t row_stride = (int64_t)nx * 4;
    // lane's fixed offset inside a footprint: plane (g & 3) of quad (g >> 2), column t
    const int64_t lane_off = (int64_t)(g >> 2) * quad_stride + t * 4 + (g & 3);
    const bool pair_ok = ((n_cells & 1) == 0) && (!grid2d || (row_len & 1) == 0);

    // ---- distinct footprints of the warp (plane independent).  32 consecutive cells of a dense map
    // cover one to three image pixels along the row (four at a corner of 2 x 2 pixels): up to four footprints
    // are kept for the pipelined path; more (a map coarser than the launcher's density rule expects) take the
    // general path at the end.
    uint32_t org0 = 0xffffffffu, org1 = 0xffffffffu, org2 = 0xffffffffu, org3 = 0xffffffffu;
    uint32_t mine = 0;     // bit 4 f + i: this lane's cell of tile i reads footprint f
    uint32_t tiles = 0;    // (uniform) bit 4 f + i: tile i has cells of footprint f;
                           // bit 16 + i: every valid cell of tile i reads ONE footprint (no masking needed)
    bool simple = true;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint32_t todo = valid_mask[i];
        while (todo) {
            const int leader = __ffs(todo) - 1;
            const uint32_t members = __shfl_sync(kFull, cls[i], leader);
            const uint32_t org = __shfl_sync(kFull, origin[i], leader);
            const uint32_t me = (members >> lane) & 1u;
            if (members == valid_mask[i]) tiles |= 1u << (16 + i);
            if (org0 == 0xffffffffu || org == org0) {
                org0 = org;
                mine |= me << i;
                tiles |= 1u << i;
            } else if (org1 == 0xffffffffu || org == org1) {
                org1 = org;
                mine |= me << (4 + i);
                tiles |= 1u << (4 + i);
            } else if (org2 == 0xffffffffu || org == org2) {
                org2 = org;
                mine |= me << (8 + i);
                tiles |= 1u << (8 + i);
            } else if (org3 == 0xffffffffu || org == org3) {   // the corner of 2 x 2 image pixels
                org3 = org;
                mine |= me << (12 + i);
                tiles |= 1u << (12 + i);
            } else {
                simple = false;
            }
            todo &= ~members;
        }
    }

    uint32_t ok[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};  // per tile: bit p set = plane p of the word is good, for
                                                           // this lane's two OUTPUT cells (2t, 2t + 1)
    int cur_word = -1;
    double *dst_row = out + (int64_t)(l0 + g) * n_cells + base0 + 2 * t;
    const double *pbase = coefq + (int64_t)((plane_begin + l0) >> 2) * quad_stride + lane_off;
    const bool has1 = org1 != 0xffffffffu;
    auto load_a = [&](double (&a)[4], uint32_t org, const double *pb, bool in_coef) {
        const double *p = pb + (int64_t)org * 4;
#pragma unroll
        for (int j = 0; j < 4; j++) a[j] = in_coef ? __ldg(p + j * row_stride) : 0.0;
    };
    // NaN bits of the lane's OUTPUT cells (2t, 2t + 1 of every tile) for the 32-plane word of plane
    // gl + g: OR over the (up to) four pixels of _should_propagate_nan_to_map.  The eight lanes
    // sharing t split the loads: lane (g, t) reads neighbour pixel (g & 3) of cell 2t + (g >> 2), two
    // xor-shuffles OR the neighbours, a third swaps the two cells: one load per tile and word.
    uint32_t pixel[4];  // that neighbour's pixel index; 0xffffffff: cell not valid
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int src = 4 * (2 * t + (g >> 2));
        const uint32_t nb = __shfl_sync(kFull, nbp[i], src);
        const bool v = (valid_mask[i] >> src) & 1u;
        const uint32_t x0 = nb & 0x3fff, y0 = (nb >> 14) & 0x3fff;
        const uint32_t dx = (g & 1) ? ((nb >> 28) & 1u) : 0u, dy = (g & 2) ? ((nb >> 29) & 1u) : 0u;
        pixel[i] = v ? (y0 + dy) * (uint32_t)nx + x0 + dx : 0xffffffffu;
    }
    auto refresh_ok = [&](int word) {
        word = min(word, n_words - 1);  // lanes past the last plane never store
        const uint32_t skip = __ldg(plane_bits + word);
        const bool consult = propagate && __ldg(plane_bits + n_words + word);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            uint32_t w = 0;
            if (consult && pixel[i] != 0xffffffffu) w = __ldg(nanbits + (int64_t)pixel[i] * n_words + word);
            w |= __shfl_xor_sync(kFull, w, 4);
            w |= __shfl_xor_sync(kFull, w, 8);
            const uint32_t good = pixel[i] != 0xffffffffu ? ~(w | skip) : 0u;
            const uint32_t other = __shfl_xor_sync(kFull, good, 16);
            ok[i][0] = (g >> 2) ? other : good;
            ok[i][1] = (g >> 2) ? good : other;
        }
    };

    // ---- pipelined path: at most four distinct footprints in the warp
    if (simple) {
        // A footprint of one plane tile is 8 planes x 4 rows x 4 columns = 1 KB = 64 chunks of 16 bytes in the
        // plane-quad layout ([quad][y][x][4 planes]: chunk c = ((q * 4 + y) * 4 + x) * 2 + half).  Lane L
        // copies chunks L (quad 0) and L + 32 (quad 1) with two 16-byte cp.async - a quarter of a kilobyte per
        // instruction and ONE address per footprint - and reads back the element of its own MMA row / column,
        // which other lanes copied: __syncwarp() after the wait makes the copies visible inside the warp.
        //
        // Each warp owns kCubicSlots footprint slots of 1 KB, used as a ring of DEPTH = kCubicSlots / NF plane
        // tiles for a warp with NF distinct footprints: the common single-footprint warp keeps five tiles in
        // flight behind the one being multiplied (an L2 round trip under a full store stream is ~4 tile times),
        // a three-footprint warp one, a four-footprint warp (a corner of 2 x 2 image pixels) none.
        __shared__ __align__(16) double stage[kCubicBlock / 32][kCubicSlots][128];
        const bool full_tiles = ncols[0] == 8 && ncols[1] == 8 && ncols[2] == 8 && ncols[3] == 8;
        const bool fast_store = full_tiles && pair_ok;
        const int n_it = (l1 - l0 + 7) / 8;
        const int nf = org3 != 0xffffffffu ? 4 : (org2 != 0xffffffffu ? 3 : (has1 ? 2 : 1));
        const int warp = threadIdx.x >> 5;
        // source of this lane's chunk inside a footprint whose top-left coefficient is at `base`:
        // row (lane >> 3) & 3, column (lane >> 1) & 3, half lane & 1 of quad 0
        const int64_t chunk_off = (int64_t)((lane >> 3) & 3) * row_stride + ((lane >> 1) & 3) * 4 + (lane & 1) * 2;
        const double *q0 = coefq + (int64_t)((plane_begin + l0) >> 2) * quad_stride + (int64_t)org0 * 4 + chunk_off;
        // footprints 1 and 2 as element offsets from footprint 0 (they fit 32 bits: nx, ny < 16384)
        const int d1 = nf > 1 ? ((int)org1 - (int)org0) * 4 : 0, d2 = nf > 2 ? ((int)org2 - (int)org0) * 4 : 0;
        const int d3 = nf > 3 ? ((int)org3 - (int)org0) * 4 : 0;
        const int64_t tile_stride = 2 * quad_stride;
        // quads of coefficients that exist from this group's first plane on (the last tile may have one)
        const int quads_ahead = (n_planes_padded - (plane_begin + l0)) >> 2;
        double *const my_chunk = &stage[warp][0][2 * lane];            // + 64 doubles: the quad-1 chunk
        const double *const my_elem = &stage[warp][0][(g >> 2) * 64 + t * 4 + (g & 3)];   // + 16 j: row j
        uint32_t clean = 0;   // (uniform) bit b: the 8 planes b*8.. of the current NaN word are good in every cell of the warp

        // refresh_ok split in two so that the loads run one 32-plane word ahead of their use
        uint32_t nw[4], nskip = 0;
        auto fetch_ok = [&](int word) {
            word = min(word, n_words - 1);
            nskip = __ldg(plane_bits + word);
            const bool consult = propagate && __ldg(plane_bits + n_words + word);
#pragma unroll
            for (int i = 0; i < 4; i++)
                nw[i] = (consult && pixel[i] != 0xffffffffu) ? __ldg(nanbits + (int64_t)pixel[i] * n_words + word) : 0u;
        };
        auto apply_ok = [&]() {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                uint32_t w = nw[i];
                w |= __shfl_xor_sync(kFull, w, 4);
                w |= __shfl_xor_sync(kFull, w, 8);
                const uint32_t good = pixel[i] != 0xffffffffu ? ~(w | nskip) : 0u;
                const uint32_t other = __shfl_xor_sync(kFull, good, 16);
                ok[i][0] = (g >> 2) ? other : good;
                ok[i][1] = (g >> 2) ? good : other;
            }
        };
        auto pipeline = [&](auto nf_tag) {
            constexpr int NF = decltype(nf_tag)::value;
            constexpr int DEPTH = kCubicSlots / NF;   // plane tiles in the ring
            static_assert(DEPTH >= 1, "a ring entry must hold every footprint of a plane tile");
            constexpr int kTile = NF * 128;           // doubles per ring entry
            int issued = 0, issue_slot = 0;
            auto issue = [&]() {
                if (issued < n_it) {
                    double *dst = my_chunk + issue_slot * kTile;
                    // the second quad of the last tile may lie past the array: copy the first one again (its rows
                    // of D are never stored, and the rows of the product are independent)
                    const int64_t second = 2 * issued + 1 < quads_ahead ? quad_stride : 0;
                    cp_async16(dst, q0);
                    cp_async16(dst + 64, q0 + second);
                    if (NF > 1) {
                        cp_async16(dst + 128, q0 + d1);
                        cp_async16(dst + 128 + 64, q0 + d1 + second);
                    }
                    if (NF > 2) {
                        cp_async16(dst + 256, q0 + d2);
                        cp_async16(dst + 256 + 64, q0 + d2 + second);
                    }
                    if (NF > 3) {
                        cp_async16(dst + 384, q0 + d3);
                        cp_async16(dst + 384 + 64, q0 + d3 + second);
                    }
                    if (2 * issued + 2 < quads_ahead) q0 += tile_stride;
                }
                issued++;
                issue_slot = issue_slot + 1 == DEPTH ? 0 : issue_slot + 1;
                cp_async_commit();  // one group per plane tile, empty past the end: uniform accounting
            };
#pragma unroll
            for (int k = 0; k < DEPTH - 1; k++) issue();
            fetch_ok((plane_begin + l0) >> 5);
            int use_slot = 0;
            for (int it = 0; it < n_it; it++) {
                const int l = l0 + 8 * it;
                const int gl = plane_begin + l;  // global plane of row 0 of this plane tile (a multiple of 8)
                __syncwarp();                    // every lane has read the ring entry this issue() overwrites (tile it - 1)
                issue();
                const int word = gl >> 5;        // the same for the 8 planes of the tile
                if (word != cur_word) {          // uniform: changes once per 32 planes
                    cur_word = word;
                    apply_ok();                  // the words fetched four tiles ago ...
                    fetch_ok(word + 1);          // ... and the next ones, consumed four tiles from now
                    uint32_t all = ok[0][0] & ok[0][1] & ok[1][0] & ok[1][1] & ok[2][0] & ok[2][1] & ok[3][0] & ok[3][1];
                    all = __reduce_and_sync(kFull, all);
                    clean = (((all & 0xffu) == 0xffu) ? 1u : 0u) | (((all & 0xff00u) == 0xff00u) ? 2u : 0u) |
                            (((all & 0xff0000u) == 0xff0000u) ? 4u : 0u) | (((all >> 24) == 0xffu) ? 8u : 0u);
                }
                cp_async_wait<DEPTH - 1>();  // this lane's chunks of plane tile `it` have landed ...
                __syncwarp();                // ... and so have the other lanes'
                const double *src = my_elem + use_slot * kTile;
                use_slot = use_slot + 1 == DEPTH ? 0 : use_slot + 1;
                double d[4][2];
#pragma unroll
                for (int i = 0; i < 4; i++) d[i][0] = d[i][1] = 0.0;
                if (NF == 1) {
                    // every valid cell reads footprint 0 and invalid cells carry zero weights: no masks
                    double a[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) a[j] = src[16 * j];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
#pragma unroll
                        for (int i = 0; i < 4; i++) dmma8x8x4(d[i][0], d[i][1], a[j], bw[i][j]);
                    }
                } else {
#pragma unroll 1
                    for (int f = 0; f < NF; f++) {   // rolled: the footprint only enters through bit positions
                        double a[4];
#pragma unroll
                        for (int j = 0; j < 4; j++) a[j] = src[f * 128 + 16 * j];
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            if (tiles & (1u << (4 * f + i))) {
                                const bool keep = (tiles & (1u << (16 + i))) || ((mine >> (4 * f + i)) & 1u);
#pragma unroll
                                for (int j = 0; j < 4; j++) dmma8x8x4(d[i][0], d[i][1], a[j], keep ? bw[i][j] : 0.0);
                            }
                        }
                    }
                }
                // ---- store: lane holds plane gl + g, cells 2t, 2t + 1 of every tile
                if (l + g < l1 && l + g >= lead) {
                    const int sh = (gl + g) & 31;
                    const bool tile_clean = (clean >> ((gl >> 3) & 3)) & 1u;   // uniform: no NaN in these 8 planes
                    auto store_tiles = [&](const int64_t step, const bool all_pairs, const bool select) {
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const double o0 = (!select || ((ok[i][0] >> sh) & 1u)) ? d[i][0] : nan;
                            const double o1 = (!select || ((ok[i][1] >> sh) & 1u)) ? d[i][1] : nan;
                            double *dst = dst_row + i * step;
                            if (all_pairs || (pair_ok && 2 * t + 1 < ncols[i])) {
                                asm volatile("st.global.cs.v2.f64 [%0], {%1, %2};" ::"l"(dst), "d"(o0), "d"(o1) : "memory");
                            } else {
                                if (2 * t < ncols[i]) __stcs(dst, o0);
                                if (2 * t + 1 < ncols[i]) __stcs(dst + 1, o1);
                            }
                        }
                    };
                    // the usual case - full tiles of consecutive cells, aligned pairs - is straight-line code
                    // whose tile offsets are immediates of the stores; tiles without a NaN skip the selects
                    if (fast_store && !grid2d) {
                        if (tile_clean)
                            store_tiles(8, true, false);
                        else
                            store_tiles(8, true, true);
                    } else if (fast_store) {
                        store_tiles(tile_step, true, true);
                    } else {
                        store_tiles(tile_step, false, true);
                    }
                }
                dst_row += 8 * n_cells;
            }
        };
        if (nf == 1)
            pipeline(std::integral_constant<int, 1>{});
        else if (nf == 2)
            pipeline(std::integral_constant<int, 2>{});
        else if (nf == 3)
            pipeline(std::integral_constant<int, 3>{});
        else
            pipeline(std::integral_constant<int, 4>{});   // one ring entry: no tile in flight, but the same staged loads
        return;
    }

    // ---- general path (four or more footprints in the warp): one pass per distinct footprint
    // among each tile's cells
    for (int l = l0; l < l1; l += 8) {
        const int gl = plane_begin + l;  // global plane of row 0 of this plane tile (multiple of 4)
        const int word = (gl + g) >> 5;
        if (word != cur_word) {  // changes at most once per 32 planes (per lane: planes gl + g)
            cur_word = word;
            refresh_ok(word);
        }
        double d[4][2];
#pragma unroll
        for (int i = 0; i < 4; i++) d[i][0] = d[i][1] = 0.0;
        const bool in_coef = (gl + g) < n_planes_padded;
        {
            uint32_t a_origin = 0xffffffffu;
            double a[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
            for (int i = 0; i < 4; i++) {
                uint32_t todo = valid_mask[i];
                while (todo) {
                    const int leader = __ffs(todo) - 1;
                    const uint32_t members = __shfl_sync(kFull, cls[i], leader);
                    const uint32_t org = __shfl_sync(kFull, origin[i], leader);
                    if (org != a_origin) {
                        a_origin = org;
                        load_a(a, org, pbase, in_coef);
                    }
                    const bool member = (members >> lane) & 1u;
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma8x8x4(d[i][0], d[i][1], a[j], member ? bw[i][j] : 0.0);
                    todo &= ~members;
                }
            }
        }
        // ---- store: lane holds plane gl + g, cells 2t, 2t + 1 of every tile
        if (l + g < l1 && l + g >= lead) {
            const int sh = (gl + g) & 31;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const double o0 = ((ok[i][0] >> sh) & 1u) ? d[i][0] : nan;
                const double o1 = ((ok[i][1] >> sh) & 1u) ? d[i][1] : nan;
                double *dst = dst_row + i * tile_step;
                if (pair_ok && 2 * t + 1 < ncols[i]) {
                    asm volatile("st.global.cs.v2.f64 [%0], {%1, %2};" ::"l"(dst), "d"(o0), "d"(o1) : "memory");
                } else {
                    if (2 * t < ncols[i]) __stcs(dst, o0);
                    if (2 * t + 1 < ncols[i]) __stcs(dst + 1, o1);
                }
            }
        }
        pbase += 2 * quad_stride;
        dst_row += 8 * n_cells;
    }
}

// ---------------------------------------------------------------------------------
// Grouped gather for a time series (pm_gather_grouped): map g of n_maps serves the planes
// [g * plane_stride, g * plane_stride + planes_per_map) of the cube; out [n_maps][planes_per_map][n_cells].
// Grid (cell blocks, map, plane group).  Per cell the weights and NaN-test pixels are set up once for the
// map and reused for every plane of the group, and every voxel takes the arithmetic of gather_nearest_kernel /
// gather_spline_kernel, so a group equals pm_gather of the same planes through the same map bit for bit.
// kQuads: groups start on a plane quad (plane_stride a multiple of 4) and are read a quad per 32-byte load;
// otherwise every plane is read from its lane of the quad (one image per epoch packed four to a quad:
// planes_per_map = plane_stride = 1, which is pm_gather_paired).
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGatherBlock)
    gather_grouped_nearest_kernel(const double *__restrict__ cube, int ny, int nx, int planes_per_map,
                                  int plane_stride, const double *__restrict__ xmaps, const double *__restrict__ ymaps,
                                  int64_t map_stride, int64_t n_cells, double *__restrict__ out, int planes_per_group) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= n_cells) return;
    const int g = blockIdx.y;
    const int l0 = blockIdx.z * planes_per_group;
    const int l1 = min(l0 + planes_per_group, planes_per_map);
    nearest_cell_planes(cube, ny, nx, g * plane_stride, l0, l1, xmaps + (int64_t)g * map_stride,
                        ymaps + (int64_t)g * map_stride, cell, n_cells, out + (int64_t)g * planes_per_map * n_cells);
}

template <int KY, int KX, bool kQuads, int kMinBlocks>
__global__ void __launch_bounds__(kGatherBlock, kMinBlocks)
    gather_grouped_kernel(const double *__restrict__ coefq, const uint32_t *__restrict__ nanbits,
                          const uint32_t *__restrict__ plane_bits, int n_words, int ny, int nx, int planes_per_map,
                          int plane_stride, const double *__restrict__ xmaps, const double *__restrict__ ymaps,
                          int64_t map_stride, int64_t n_cells, uint32_t flags, double *__restrict__ out,
                          int planes_per_group) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= n_cells) return;
    const int g = blockIdx.y;
    const int l0 = blockIdx.z * planes_per_group;  // multiple of 4
    const int l1 = min(l0 + planes_per_group, planes_per_map);
    const bool propagate = (flags & PM_FLAG_PROPAGATE_NAN) != 0;
    const int64_t m = (int64_t)g * map_stride + cell;
    CellState<KY, KX> cs;
    setup_cell<KY, KX>(cs, __ldg(xmaps + m), __ldg(ymaps + m), ny, nx, propagate);
    out += (int64_t)g * planes_per_map * n_cells;
    if (kQuads) {
        spline_cell_quads<KY, KX>(cs, coefq, nanbits, plane_bits, n_words, ny, nx, g * plane_stride, l0, l1,
                                  propagate, cell, n_cells, out);
    } else {
        double *dst = out + (int64_t)l0 * n_cells + cell;
        for (int l = l0; l < l1; l++, dst += n_cells)
            __stcs(dst, spline_cell_plane<KY, KX>(cs, coefq, nanbits, plane_bits, n_words, ny, nx,
                                                  g * plane_stride + l, propagate));
    }
}

// launch_gather's switch to the DMMA kernel for cubic: many map cells per image pixel share a footprint.
// Measured crossover with the one-cell-per-thread kernel (tools/probe_density.py): ~16 map cells per image
// pixel - at 15.8 the scalar kernel is 10 % faster, at 63 the DMMA kernel 1.5x, at 400 (BASELINE C4) 2x
static bool dense_map(int64_t n_cells, int ny, int nx) {
    return n_cells >= (int64_t)20 * nx * ny && nx < 16384 && ny < 16384;
}

cudaError_t launch_gather(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes,
                          int ny, int nx, int plane_begin, int plane_count, const double *xmap, const double *ymap,
                          int64_t n_cells, int64_t cells_per_row, int mode, uint32_t flags, double *out, int sm_count,
                          cudaStream_t st) {
    (void)sm_count;
    if (n_cells == 0 || plane_count == 0) return cudaSuccess;
    int ppg = 128;  // planes per CTA: amortises the per-cell weights, bounds CTA run time
    if (plane_count < ppg) ppg = (plane_count + 3) / 4 * 4;
    // every CTA of the scalar kernels covers kGatherBlock cells (the DMMA kernel sizes its own grid below)
    dim3 grid((unsigned)((n_cells + kGatherBlock - 1) / kGatherBlock), (unsigned)((plane_count + ppg - 1) / ppg));
    const int n_words = (n_planes + 31) / 32;
    int ky = mode, kx = mode;  // spline degree along image rows (y) / columns (x)
    if (mode & PM_INTERP_MIXED) {
        ky = (mode >> 4) & 0xF;
        kx = mode & 0xF;
    }
    if (mode == PM_INTERP_NEAREST) {
        gather_nearest_kernel<<<grid, kGatherBlock, 0, st>>>(src, ny, nx, plane_begin, plane_count, xmap, ymap, n_cells,
                                                             out, ppg);
        count_launches(1);
        return cudaGetLastError();
    }
    if (ky < 1 || ky > 3 || kx < 1 || kx > 3) return cudaErrorInvalidValue;
#define PM_SPLINE(KY, KX, MB)                                                                                     \
    gather_spline_kernel<KY, KX, MB><<<grid, kGatherBlock, 0, st>>>(src, nanbits, plane_bits, n_words, ny, nx,    \
                                                                    plane_begin, plane_count, xmap, ymap, n_cells, \
                                                                    flags, out, ppg)
    static const int v = tune_int("PM_CUBIC_VARIANT", -1);
    // dense maps (many cells per image pixel share a footprint): warp-tiled DMMA kernel
    const bool dense = dense_map(n_cells, ny, nx);
    if (ky == 3 && kx == 3 && v != 0 && (dense || v > 0)) {
        // larger plane groups: the per-warp setup (map loads, weights, footprint classes) is heavier here
        // than in the scalar kernel
        static const int mma_ppg = tune_int("PM_MMA_PPG", 512);
        // the kernel wants plane tiles aligned to 8 planes (see its header): a range starting on an odd quad is
        // launched from the quad before it, whose four planes are computed and dropped
        const int lead = plane_begin & 7;   // 0 or 4 (plane_begin is a multiple of 4)
        const int pb = plane_begin - lead, pc = plane_count + lead;
        const int g2 = pc < mma_ppg ? (pc + 7) / 8 * 8 : mma_ppg;
        // map row length known and regular -> 4 x 8 cell blocks per warp, else 32 consecutive cells
        // (measured on C4: for long rows the 1-D order is ~4 % faster - longer contiguous store
        // runs - so the blocks are only used when a warp's 32 cells would wrap across map rows)
        const bool rows_ok = cells_per_row > 0 && cells_per_row < 64 && cells_per_row < n_cells &&
                             n_cells % cells_per_row == 0;
        const int64_t row_len = rows_ok ? cells_per_row : n_cells;
        const int64_t n_warps = rows_ok ? ((n_cells / row_len + 3) / 4) * ((row_len + 7) / 8) : (n_cells + 31) / 32;
        dim3 grid2((unsigned)((n_warps + kCubicBlock / 32 - 1) / (kCubicBlock / 32)),
                   (unsigned)((pc + g2 - 1) / g2));
        gather_cubic_mma_kernel<<<grid2, kCubicBlock, 0, st>>>(src, nanbits, plane_bits, n_words, ny, nx,
                                                                (n_planes + 3) / 4 * 4, pb, pc, xmap, ymap, n_cells,
                                                                row_len, flags, out - (int64_t)lead * n_cells, g2,
                                                                lead);
    } else {
        switch (ky * 4 + kx) {
            case 1 * 4 + 1: PM_SPLINE(2, 2, 5); break;
            case 1 * 4 + 2: PM_SPLINE(2, 3, 3); break;
            case 1 * 4 + 3: PM_SPLINE(2, 4, 3); break;
            case 2 * 4 + 1: PM_SPLINE(3, 2, 3); break;
            case 2 * 4 + 2: PM_SPLINE(3, 3, 3); break;
            case 2 * 4 + 3: PM_SPLINE(3, 4, 2); break;
            case 3 * 4 + 1: PM_SPLINE(4, 2, 3); break;
            case 3 * 4 + 2: PM_SPLINE(4, 3, 2); break;
            default: PM_SPLINE(4, 4, 2); break;
        }
    }
#undef PM_SPLINE
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_gather_grouped(const double *src, const uint32_t *nanbits, const uint32_t *plane_bits, int n_planes,
                                  int ny, int nx, int n_maps, int planes_per_map, int plane_stride, const double *xmaps,
                                  const double *ymaps, int64_t map_stride, int64_t n_cells, int mode, uint32_t flags,
                                  double *out, int sm_count, cudaStream_t st) {
    if (n_maps == 0 || planes_per_map == 0 || n_cells == 0) return cudaSuccess;
    int ppg = 128;  // planes per CTA, as launch_gather
    if (planes_per_map < ppg) ppg = (planes_per_map + 3) / 4 * 4;
    const dim3 grid((unsigned)((n_cells + kGatherBlock - 1) / kGatherBlock), (unsigned)n_maps,
                    (unsigned)((planes_per_map + ppg - 1) / ppg));
    if (mode == PM_INTERP_NEAREST) {
        gather_grouped_nearest_kernel<<<grid, kGatherBlock, 0, st>>>(src, ny, nx, planes_per_map, plane_stride, xmaps,
                                                                     ymaps, map_stride, n_cells, out, ppg);
        count_launches(1);
        return cudaGetLastError();
    }
    int ky = mode, kx = mode;
    if (mode & PM_INTERP_MIXED) {
        ky = (mode >> 4) & 0xF;
        kx = mode & 0xF;
    }
    if (ky < 1 || ky > 3 || kx < 1 || kx > 3) return cudaErrorInvalidValue;
    const bool quads = planes_per_map > 1 && plane_stride % 4 == 0;
    if (ky == 3 && kx == 3 && quads && dense_map(n_cells, ny, nx)) {
        // a cube per map on a dense map: pm_gather's own DMMA launch per map, so each group is its result bit
        // for bit (plane_begin = g * plane_stride is a multiple of 4)
        for (int g = 0; g < n_maps; g++) {
            const cudaError_t e = launch_gather(src, nanbits, plane_bits, n_planes, ny, nx, g * plane_stride,
                                                planes_per_map, xmaps + (int64_t)g * map_stride,
                                                ymaps + (int64_t)g * map_stride, n_cells, 0, mode, flags,
                                                out + (int64_t)g * planes_per_map * n_cells, sm_count, st);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    const int n_words = (n_planes + 31) / 32;
    // CTAs per SM (quad form, plane-by-plane form): the most at which each instantiation compiles without spills
    // (ptxas -v); the quad form carries the group indexing on top of gather_spline_kernel's state
#define PM_GROUPED(KY, KX, MBQ, MB)                                                                                    \
    do {                                                                                                            \
        if (quads)                                                                                                  \
            gather_grouped_kernel<KY, KX, true, MBQ><<<grid, kGatherBlock, 0, st>>>(                                 \
                src, nanbits, plane_bits, n_words, ny, nx, planes_per_map, plane_stride, xmaps, ymaps, map_stride,  \
                n_cells, flags, out, ppg);                                                                          \
        else                                                                                                        \
            gather_grouped_kernel<KY, KX, false, MB><<<grid, kGatherBlock, 0, st>>>(                                \
                src, nanbits, plane_bits, n_words, ny, nx, planes_per_map, plane_stride, xmaps, ymaps, map_stride,  \
                n_cells, flags, out, ppg);                                                                          \
    } while (0)
    switch (ky * 4 + kx) {
        case 1 * 4 + 1: PM_GROUPED(2, 2, 4, 6); break;
        case 1 * 4 + 2: PM_GROUPED(2, 3, 3, 3); break;
        case 1 * 4 + 3: PM_GROUPED(2, 4, 2, 3); break;
        case 2 * 4 + 1: PM_GROUPED(3, 2, 2, 3); break;
        case 2 * 4 + 2: PM_GROUPED(3, 3, 2, 3); break;
        case 2 * 4 + 3: PM_GROUPED(3, 4, 2, 2); break;
        case 3 * 4 + 1: PM_GROUPED(4, 2, 2, 3); break;
        case 3 * 4 + 2: PM_GROUPED(4, 3, 2, 2); break;
        default: PM_GROUPED(4, 4, 2, 2); break;
    }
#undef PM_GROUPED
    count_launches(1);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------
// spline preparation
// ---------------------------------------------------------------------------------
struct PlaneStats {
    long long n_nan;
    long long n_bad;
    long long n_iso;   // bad pixels whose nine (edge-clamped) neighbours are all bad: the only ones the median fills
};

// Planes of a cube are small (C4: 64 x 64) and many, planes of a time series are large (C5:
// 1024 x 1024) and few per batch: a plane is spread over `gridDim.y` CTAs so that both shapes
// fill the machine.
// pass 1: NaN mask, bad-pixel counts (atomically into zeroed `stats`), copy into the coefficient buffer
__global__ void __launch_bounds__(256) classify_kernel(const double *__restrict__ cube, int64_t plane_px,
                                                       double *__restrict__ coef, PlaneStats *__restrict__ stats) {
    const int l = blockIdx.x;
    const double *src = cube + (int64_t)l * plane_px;
    double *dst = coef + (int64_t)l * plane_px;
    long long n_nan = 0, n_bad = 0;
    for (int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; i < plane_px; i += (int64_t)gridDim.y * blockDim.x) {
        double v = src[i];
        bool isn = isnan(v);
        n_nan += isn;
        n_bad += !isfinite(v);
        dst[i] = v;
    }
    __shared__ long long s_nan[256], s_bad[256];
    s_nan[threadIdx.x] = n_nan;
    s_bad[threadIdx.x] = n_bad;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            s_nan[threadIdx.x] += s_nan[threadIdx.x + o];
            s_bad[threadIdx.x] += s_bad[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && (s_nan[0] | s_bad[0])) {
        atomicAdd(reinterpret_cast<unsigned long long *>(&stats[l].n_nan), (unsigned long long)s_nan[0]);
        atomicAdd(reinterpret_cast<unsigned long long *>(&stats[l].n_bad), (unsigned long long)s_bad[0]);
    }
}
__global__ void plane_flags_kernel(const PlaneStats *__restrict__ stats, int n_planes, int64_t plane_px,
                                   uint8_t *__restrict__ plane_skip) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_planes) return;
    uint8_t flag = 0;
    if (stats[l].n_nan == plane_px) flag |= kPlaneAllNan;
    if (stats[l].n_nan > 0) flag |= kPlaneHasNan;
    plane_skip[l] = flag;
}

__device__ __forceinline__ unsigned long long order_key(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_to_double(unsigned long long k) {
    unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// k-th smallest (0-based) finite value of a plane: MSB-first radix select, one CTA
__device__ double radix_select(const double *__restrict__ src, int64_t n, long long k) {
    __shared__ unsigned int hist[256];
    __shared__ unsigned long long s_prefix, s_mask;
    __shared__ long long s_k;
    if (threadIdx.x == 0) {
        s_prefix = 0;
        s_mask = 0;
        s_k = k;
    }
    __syncthreads();
    for (int pass = 7; pass >= 0; pass--) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        const unsigned long long prefix = s_prefix, mask = s_mask;
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
            double v = src[i];
            if (isfinite(v)) {
                unsigned long long key = order_key(v);
                if ((key & mask) == prefix) atomicAdd(&hist[(key >> (8 * pass)) & 255ull], 1u);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            long long kk = s_k, cum = 0;
            int b = 0;
            for (; b < 256; b++) {
                if (cum + (long long)hist[b] > kk) break;
                cum += hist[b];
            }
            if (b > 255) b = 255;
            s_k = kk - cum;
            s_prefix = prefix | ((unsigned long long)b << (8 * pass));
            s_mask = mask | (0xffull << (8 * pass));
        }
        __syncthreads();
    }
    double r = key_to_double(s_prefix);
    __syncthreads();
    return r;
}

// pass 2: np.nanmedian of the finite pixels of each plane that has bad pixels
__global__ void __launch_bounds__(256) median_kernel(const double *__restrict__ cube, int64_t plane_px,
                                                     const PlaneStats *__restrict__ stats,
                                                     double *__restrict__ median) {
    const int l = blockIdx.x;
    const long long n_bad = stats[l].n_bad;
    if (stats[l].n_iso == 0) return;  // no pixel takes the median (uniform for the CTA)
    const long long m = plane_px - n_bad;
    double med = 0.0;  // np.all(bad) -> 0.0 (body_xy.py:1890-1891)
    if (m > 0) {
        const double *src = cube + (int64_t)l * plane_px;
        if (m & 1) {
            med = radix_select(src, plane_px, m / 2);
        } else {
            double a = radix_select(src, plane_px, m / 2 - 1);
            double b = radix_select(src, plane_px, m / 2);
            med = (a + b) / 2.0;
        }
    }
    if (threadIdx.x == 0) median[l] = med;
}

// pass 2 for LARGE planes: the same MSB-first radix select with the histogram of every pass built
// by many CTAs per plane (shared-memory histogram per CTA, merged with global atomics) and the
// bucket chosen by a one-thread-per-plane kernel in between: 1 + 2 x 8 small launches that each
// stream the batch once, instead of one CTA walking a megapixel plane sixteen times.
// 11-bit digits: six passes over the batch instead of eight with bytes (the last digit has 9 bits)
constexpr int kSelBits = 11, kSelBins = 1 << kSelBits, kSelPasses = 6;
__host__ __device__ __forceinline__ int sel_shift(int pass) { return pass == 0 ? 0 : 64 - kSelBits * (kSelPasses - pass); }
__host__ __device__ __forceinline__ unsigned sel_width_mask(int pass) { return pass == 0 ? (1u << 9) - 1u : (unsigned)kSelBins - 1u; }

struct SelectState {
    unsigned long long prefix[2], mask;
    long long k[2];
    int n_sel;  // 0: nothing to select, 1: odd count (one order statistic), 2: even count (two)
};
__global__ void select_init_kernel(const PlaneStats *__restrict__ stats, int n_planes, int64_t plane_px,
                                   SelectState *__restrict__ state, unsigned int *__restrict__ hist,
                                   double *__restrict__ median) {
    const int l = blockIdx.x;
    for (int i = threadIdx.x; i < 2 * kSelBins; i += blockDim.x) hist[(int64_t)l * 2 * kSelBins + i] = 0;
    if (threadIdx.x != 0) return;
    SelectState st;
    st.prefix[0] = st.prefix[1] = st.mask = 0;
    st.k[0] = st.k[1] = 0;
    st.n_sel = 0;
    const long long n_bad = stats[l].n_bad, m = plane_px - n_bad;
    if (stats[l].n_iso > 0) {   // the median is only ever written into isolated bad pixels: skip it otherwise
        if (m <= 0) {
            median[l] = 0.0;  // np.all(bad) -> 0.0 (body_xy.py:1890-1891)
        } else if (m & 1) {
            st.n_sel = 1;
            st.k[0] = m / 2;
        } else {
            st.n_sel = 2;
            st.k[0] = m / 2 - 1;
            st.k[1] = m / 2;
        }
    }
    state[l] = st;
}
__global__ void __launch_bounds__(256) select_hist_kernel(const double *__restrict__ cube, int64_t plane_px,
                                                          const SelectState *__restrict__ state,
                                                          unsigned int *__restrict__ hist, int pass) {
    const int l = blockIdx.x;
    const SelectState st = state[l];
    if (st.n_sel == 0) return;  // uniform for the CTA
    __shared__ unsigned int sh[2][kSelBins];
    for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) {
        sh[0][i] = 0;
        sh[1][i] = 0;
    }
    __syncthreads();
    const double *src = cube + (int64_t)l * plane_px;
    const bool same = st.n_sel == 2 && st.prefix[0] == st.prefix[1];  // both statistics still in one bucket
    const int shift = sel_shift(pass);
    const unsigned wmask = sel_width_mask(pass);
    for (int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; i < plane_px; i += (int64_t)gridDim.y * blockDim.x) {
        const double v = src[i];
        if (isfinite(v)) {
            const unsigned long long key = order_key(v);
            const unsigned d = (unsigned)(key >> shift) & wmask;
            if ((key & st.mask) == st.prefix[0]) atomicAdd(&sh[0][d], 1u);
            if (st.n_sel == 2 && !same && (key & st.mask) == st.prefix[1]) atomicAdd(&sh[1][d], 1u);
        }
    }
    __syncthreads();
    unsigned int *g = hist + (int64_t)l * 2 * kSelBins;
    for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) {
        if (sh[0][i]) atomicAdd(&g[i], sh[0][i]);
        const unsigned int second = same ? sh[0][i] : sh[1][i];
        if (st.n_sel == 2 && second) atomicAdd(&g[kSelBins + i], second);
    }
}
// one warp per plane: lane i owns buckets kPer i .. kPer i + kPer - 1; the bucket holding rank k is
// found from the warp prefix sum of the lane totals
__global__ void __launch_bounds__(128) select_pick_kernel(SelectState *__restrict__ state,
                                                          unsigned int *__restrict__ hist, int n_planes, int pass,
                                                          double *__restrict__ median) {
    constexpr int kPer = kSelBins / 32;
    const int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (l >= n_planes) return;  // whole warp
    SelectState st = state[l];
    if (st.n_sel == 0) return;
    unsigned int *g = hist + (int64_t)l * 2 * kSelBins;
    const int shift = sel_shift(pass);
    for (int s = 0; s < st.n_sel; s++) {
        const unsigned int *c = g + kSelBins * s + kPer * lane;
        long long mine = 0;
        for (int b = 0; b < kPer; b++) mine += c[b];
        long long incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        const long long before = incl - mine;   // counts in the buckets below this lane's
        const bool holds = before <= st.k[s] && st.k[s] < incl;
        const unsigned owner = __ballot_sync(0xffffffffu, holds);
        int bucket = kSelBins - 1;
        long long cum = before;
        if (holds) {
            bucket = kPer * lane;
            for (int b = 0; b < kPer; b++) {
                if (cum + (long long)c[b] > st.k[s]) break;
                cum += c[b];
                bucket = kPer * lane + b + 1;
            }
        }
        const int src = owner ? __ffs(owner) - 1 : 31;   // a rank beyond the count cannot happen
        bucket = __shfl_sync(0xffffffffu, bucket, src);
        cum = __shfl_sync(0xffffffffu, cum, src);
        st.k[s] -= cum;
        st.prefix[s] |= (unsigned long long)min(bucket, (int)sel_width_mask(pass)) << shift;
    }
    st.mask |= (unsigned long long)sel_width_mask(pass) << shift;
    __syncwarp();
    for (int i = lane; i < 2 * kSelBins; i += 32) g[i] = 0;
    if (lane == 0) {
        state[l] = st;
        if (pass == 0) {
            const double a = key_to_double(st.prefix[0]);
            median[l] = st.n_sel == 1 ? a : (a + key_to_double(st.prefix[1])) / 2.0;
        }
    }
}

// pass 2: replace bad pixels that have a good neighbour by the 3 x 3 nan-mean (body_xy.py:1893-1903) and
// COUNT the others (all nine edge-clamped neighbours bad): only those take np.nanmedian of the plane
// (`cleaned[bad] = median` is overwritten everywhere else), so the median - six passes over the batch for
// megapixel planes - is computed only for planes that have such a pixel (pass 3) and written by pass 4.
__device__ __forceinline__ bool all_neighbours_bad(const double *__restrict__ img, int i, int j, int ny, int nx) {
    // uniform_filter(bad, size=3) on a bool array is True only when all nine
    // reflected neighbours are bad (SURVEY 8(a)); reflect == clamp for size 3
    bool all_bad = true;
    for (int di = -1; di <= 1; di++)
        for (int dj = -1; dj <= 1; dj++) {
            int ii = min(max(i + di, 0), ny - 1), jj = min(max(j + dj, 0), nx - 1);
            all_bad = all_bad && !isfinite(img[(int64_t)ii * nx + jj]);
        }
    return all_bad;
}
__global__ void __launch_bounds__(256) repair_kernel(const double *__restrict__ cube, int n_planes, int ny,
                                                     int nx, PlaneStats *__restrict__ stats,
                                                     double *__restrict__ coef) {
    // blockIdx.y = plane; rows are walked with 32-bit arithmetic (no 64-bit division per pixel)
    const int l = blockIdx.y;
    if (stats[l].n_bad == 0) return;
    const int64_t plane_px = (int64_t)ny * nx;
    const double *img = cube + (int64_t)l * plane_px;
    unsigned long long n_iso = 0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < plane_px; r += (int64_t)gridDim.x * blockDim.x) {
        if (isfinite(img[r])) continue;
        const int i = (int)(r / nx), j = (int)(r - (int64_t)i * nx);   // bad pixels only
        if (all_neighbours_bad(img, i, j, ny, nx)) {
            n_iso++;
            continue;
        }
        // np.nanmean over the window clipped at the image edge, inf treated as NaN
        double sum = 0.0;
        int cnt = 0;
        for (int ii = max(i - 1, 0); ii <= min(i + 1, ny - 1); ii++)
            for (int jj = max(j - 1, 0); jj <= min(j + 1, nx - 1); jj++) {
                double w = img[(int64_t)ii * nx + jj];
                if (isfinite(w)) {
                    sum += w;
                    cnt++;
                }
            }
        coef[(int64_t)l * plane_px + r] = sum / (double)cnt;
    }
    for (int o = 16; o > 0; o >>= 1) n_iso += __shfl_down_sync(0xffffffffu, n_iso, o);
    if ((threadIdx.x & 31) == 0 && n_iso)
        atomicAdd(reinterpret_cast<unsigned long long *>(&stats[l].n_iso), n_iso);
}
// pass 4: the isolated bad pixels take the plane's median
__global__ void __launch_bounds__(256) fill_isolated_kernel(const double *__restrict__ cube, int ny, int nx,
                                                            const PlaneStats *__restrict__ stats,
                                                            const double *__restrict__ median,
                                                            double *__restrict__ coef) {
    const int l = blockIdx.y;
    if (stats[l].n_iso == 0) return;
    const int64_t plane_px = (int64_t)ny * nx;
    const double *img = cube + (int64_t)l * plane_px;
    const double med = median[l];
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < plane_px; r += (int64_t)gridDim.x * blockDim.x) {
        if (isfinite(img[r])) continue;
        const int i = (int)(r / nx), j = (int)(r - (int64_t)i * nx);
        if (all_neighbours_bad(img, i, j, ny, nx)) coef[(int64_t)l * plane_px + r] = med;
    }
}

// pass 4/5: separable not-a-knot B-spline coefficient solve with a banded (2,2) LU
// lu = [l1 | l2 | d | u1 | u2], each of length n
__device__ __forceinline__ void banded_solve(double *line, int n, int64_t stride, const double *__restrict__ lu) {
    const double *l1 = lu, *l2 = lu + n, *d = lu + 2 * n, *u1 = lu + 3 * n, *u2 = lu + 4 * n;
    double ym1 = 0.0, ym2 = 0.0;
    for (int i = 0; i < n; i++) {
        double yv = line[i * stride] - l1[i] * ym1 - l2[i] * ym2;
        line[i * stride] = yv;
        ym2 = ym1;
        ym1 = yv;
    }
    double xp1 = 0.0, xp2 = 0.0;
    for (int i = n - 1; i >= 0; i--) {
        double xv = (line[i * stride] - u1[i] * xp1 - u2[i] * xp2) / d[i];
        line[i * stride] = xv;
        xp2 = xp1;
        xp1 = xv;
    }
}
__global__ void __launch_bounds__(128) prefilter_rows_kernel(double *__restrict__ coef,
                                                             const uint8_t *__restrict__ plane_skip,
                                                             int n_planes, int ny, int nx,
                                                             const double *__restrict__ lu_x) {
    const int64_t lines = (int64_t)n_planes * ny;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < lines;
         t += (int64_t)gridDim.x * blockDim.x) {
        if (plane_skip[t / ny] & kPlaneAllNan) continue;
        banded_solve(coef + t * nx, nx, 1, lu_x);
    }
}
__global__ void __launch_bounds__(128) prefilter_cols_kernel(double *__restrict__ coef,
                                                             const uint8_t *__restrict__ plane_skip,
                                                             int n_planes, int ny, int nx,
                                                             const double *__restrict__ lu_y) {
    const int64_t lines = (int64_t)n_planes * nx;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < lines;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = t / nx;
        if (plane_skip[l] & kPlaneAllNan) continue;
        const int64_t col = t - l * nx;
        banded_solve(coef + l * (int64_t)ny * nx + col, ny, nx, lu_y);
    }
}

// pass 6: pack the repaired / prefiltered planes [l][y][x] into plane quads
// [l / 4][y][x][l % 4] (zero padding up to a multiple of four planes)
__global__ void __launch_bounds__(256) pack_quads_kernel(const double *__restrict__ planes, int n_planes,
                                                         int64_t plane_px, double *__restrict__ coefq) {
    const int64_t n_quads = (n_planes + 3) / 4;
    const int64_t total = n_quads * plane_px;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = t / plane_px, px = t - q * plane_px;
        double v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int64_t l = 4 * q + j;
            v[j] = l < n_planes ? planes[l * plane_px + px] : 0.0;
        }
        double4 o = make_double4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<double4 *>(coefq + t * 4) = o;
    }
}
// pass 7: NaN bit planes [pixel][word] of the ORIGINAL cube and the per-word plane bits
__global__ void __launch_bounds__(256) pack_nanbits_kernel(const double *__restrict__ cube, int n_planes,
                                                           int64_t plane_px, int n_words,
                                                           uint32_t *__restrict__ nanbits) {
    const int64_t total = plane_px * n_words;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t wd = t / plane_px, px = t - wd * plane_px;  // consecutive threads -> consecutive pixels
        uint32_t bits = 0;
        const int lbeg = (int)wd * 32, lend = min(lbeg + 32, n_planes);
        for (int l = lbeg; l < lend; l++) bits |= (isnan(cube[(int64_t)l * plane_px + px]) ? 1u : 0u) << (l - lbeg);
        nanbits[px * n_words + wd] = bits;
    }
}
__global__ void plane_bits_kernel(const uint8_t *__restrict__ plane_skip, int n_planes, int n_words,
                                  uint32_t *__restrict__ plane_bits) {
    const int wd = blockIdx.x * blockDim.x + threadIdx.x;
    if (wd >= n_words) return;
    uint32_t skip = 0, has = 0;
    for (int l = wd * 32; l < min(wd * 32 + 32, n_planes); l++) {
        if (plane_skip[l] & kPlaneAllNan) skip |= 1u << (l - wd * 32);
        if (plane_skip[l] & kPlaneHasNan) has = 1u;
    }
    plane_bits[wd] = skip;
    plane_bits[n_words + wd] = has;
}

// host: LU factors of the collocation matrix B_j(x_i) of degree `deg` (no pivoting; it is
// totally positive); band storage fits both degrees (cubic: 2 + 2 off-diagonals,
// quadratic: 1 + 1)
static const std::vector<double> &spline_lu(int n, int deg) {
    static std::map<std::pair<int, int>, std::vector<double>> cache;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find({n, deg});
    if (it != cache.end()) return it->second;
    // band storage: A[i][j - i + 2] for |j - i| <= 2
    std::vector<double> A((size_t)n * 5, 0.0);
    for (int i = 0; i < n; i++) {
        double h[4] = {0.0, 0.0, 0.0, 0.0};
        int first = deg == 3 ? bspline_weights<3>((double)i, n, h) : bspline_weights<2>((double)i, n, h);
        for (int m = 0; m <= deg; m++) {
            int j = first + m;
            if (j < 0 || j >= n) continue;
            int off = j - i + 2;
            if (off >= 0 && off < 5) A[(size_t)i * 5 + off] = h[m];
        }
    }
    std::vector<double> lu((size_t)n * 5, 0.0);
    double *l1 = lu.data(), *l2 = l1 + n, *d = l2 + n, *u1 = d + n, *u2 = u1 + n;
    auto at = [&](int i, int j) -> double & { return A[(size_t)i * 5 + (j - i + 2)]; };
    for (int i = 0; i < n; i++) {
        for (int r = i + 1; r <= i + 2 && r < n; r++) {
            double m = at(r, i) / at(i, i);
            for (int j = i; j <= i + 2 && j < n; j++) {
                if (j - r >= -2 && j - r <= 2) at(r, j) -= m * at(i, j);
            }
            if (r == i + 1) l1[r] = m; else l2[r] = m;
        }
        d[i] = at(i, i);
        u1[i] = (i + 1 < n) ? at(i, i + 1) : 0.0;
        u2[i] = (i + 2 < n) ? at(i, i + 2) : 0.0;
    }
    return cache.emplace(std::make_pair(n, deg), std::move(lu)).first->second;
}

static inline int64_t align256(int64_t v) { return (v + 255) / 256 * 256; }

int64_t spline_coef_bytes(int n_planes, int ny, int nx) {
    return (int64_t)((n_planes + 3) / 4) * ny * nx * 4 * (int64_t)sizeof(double);
}
int64_t spline_nanbits_bytes(int n_planes, int ny, int nx) {
    return (int64_t)ny * nx * ((n_planes + 31) / 32) * (int64_t)sizeof(uint32_t);
}
int64_t spline_planebits_bytes(int n_planes) { return 2 * (int64_t)((n_planes + 31) / 32) * (int64_t)sizeof(uint32_t); }

int64_t spline_work_bytes(int n_planes, int ny, int nx, int degree) {
    int64_t b = align256((int64_t)n_planes * sizeof(PlaneStats)) + align256((int64_t)n_planes * sizeof(double)) +
                align256((int64_t)n_planes) + align256((int64_t)n_planes * ny * nx * (int64_t)sizeof(double));
    b += align256((int64_t)5 * nx * sizeof(double)) + align256((int64_t)5 * ny * sizeof(double));
    b += align256((int64_t)n_planes * sizeof(SelectState)) +
         align256((int64_t)n_planes * 2 * kSelBins * sizeof(unsigned int));
    return b;
}

cudaError_t launch_spline_prepare(const double *cube, int n_planes, int ny, int nx, int degree, double *coefq,
                                  uint32_t *nanbits, uint32_t *plane_bits, void *work, int sm_count,
                                  cudaStream_t st) {
    if (n_planes == 0) return cudaSuccess;
    char *w = static_cast<char *>(work);
    PlaneStats *stats = reinterpret_cast<PlaneStats *>(w);
    w += align256((int64_t)n_planes * sizeof(PlaneStats));
    double *median = reinterpret_cast<double *>(w);
    w += align256((int64_t)n_planes * sizeof(double));
    uint8_t *plane_skip = reinterpret_cast<uint8_t *>(w);
    w += align256((int64_t)n_planes);
    double *coef = reinterpret_cast<double *>(w);  // natural layout [l][y][x] scratch
    w += align256((int64_t)n_planes * ny * nx * (int64_t)sizeof(double));
    const int64_t plane_px = (int64_t)ny * nx;
    const int n_words = (n_planes + 31) / 32;
    // CTAs per plane: enough to fill the machine when the planes are few and large
    const int chunks = (int)std::max<int64_t>(
        1, std::min<int64_t>((plane_px + 4095) / 4096, ((int64_t)sm_count * 8 + n_planes - 1) / n_planes));
    cudaError_t me = cudaMemsetAsync(stats, 0, (size_t)n_planes * sizeof(PlaneStats), st);
    if (me != cudaSuccess) return me;
    classify_kernel<<<dim3(n_planes, chunks), 256, 0, st>>>(cube, plane_px, coef, stats);
    plane_flags_kernel<<<(n_planes + 255) / 256, 256, 0, st>>>(stats, n_planes, plane_px, plane_skip);
    count_launches(1);
    const int rblocks = (int)std::max<int64_t>(
        1, std::min<int64_t>((plane_px + 255) / 256, ((int64_t)sm_count * 16 + n_planes - 1) / n_planes));
    repair_kernel<<<dim3(rblocks, n_planes), 256, 0, st>>>(cube, n_planes, ny, nx, stats, coef);
    if (chunks == 1) {
        median_kernel<<<n_planes, 256, 0, st>>>(cube, plane_px, stats, median);
    } else {
        char *tail = static_cast<char *>(work) + spline_work_bytes(n_planes, ny, nx, degree) -
                     align256((int64_t)n_planes * sizeof(SelectState)) -
                     align256((int64_t)n_planes * 2 * kSelBins * sizeof(unsigned int));
        SelectState *state = reinterpret_cast<SelectState *>(tail);
        unsigned int *hist = reinterpret_cast<unsigned int *>(tail + align256((int64_t)n_planes * sizeof(SelectState)));
        select_init_kernel<<<n_planes, 256, 0, st>>>(stats, n_planes, plane_px, state, hist, median);
        for (int pass = kSelPasses - 1; pass >= 0; pass--) {
            select_hist_kernel<<<dim3(n_planes, chunks), 256, 0, st>>>(cube, plane_px, state, hist, pass);
            select_pick_kernel<<<(n_planes + 3) / 4, 128, 0, st>>>(state, hist, n_planes, pass, median);
        }
        count_launches(2 * kSelPasses);
    }
    fill_isolated_kernel<<<dim3(rblocks, n_planes), 256, 0, st>>>(cube, ny, nx, stats, median, coef);
    count_launches(4);
    int deg_y = degree, deg_x = degree;  // rows (image y) / columns (image x)
    if (degree & PM_INTERP_MIXED) {
        deg_y = (degree >> 4) & 0xF;
        deg_x = degree & 0xF;
    }
    {
        double *lu_x = reinterpret_cast<double *>(w);
        w += align256((int64_t)5 * nx * sizeof(double));
        double *lu_y = reinterpret_cast<double *>(w);
        int64_t rows = (int64_t)n_planes * ny, cols = (int64_t)n_planes * nx;
        int rb = (int)std::min<int64_t>((rows + 127) / 128, (int64_t)sm_count * 16);
        int cb = (int)std::min<int64_t>((cols + 127) / 128, (int64_t)sm_count * 16);
        if (deg_x >= 2) {  // solve along x (within image rows) with the column-axis degree
            const std::vector<double> &hx = spline_lu(nx, deg_x);
            cudaError_t e = cudaMemcpyAsync(lu_x, hx.data(), hx.size() * sizeof(double), cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return e;
            prefilter_rows_kernel<<<rb, 128, 0, st>>>(coef, plane_skip, n_planes, ny, nx, lu_x);
            count_launches(1);
        }
        if (deg_y >= 2) {
            const std::vector<double> &hy = spline_lu(ny, deg_y);
            cudaError_t e = cudaMemcpyAsync(lu_y, hy.data(), hy.size() * sizeof(double), cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return e;
            prefilter_cols_kernel<<<cb, 128, 0, st>>>(coef, plane_skip, n_planes, ny, nx, lu_y);
            count_launches(1);
        }
    }
    const int64_t quads_total = (int64_t)((n_planes + 3) / 4) * plane_px;
    pack_quads_kernel<<<(int)std::min<int64_t>((quads_total + 255) / 256, (int64_t)sm_count * 32), 256, 0, st>>>(
        coef, n_planes, plane_px, coefq);
    const int64_t words_total = plane_px * n_words;
    pack_nanbits_kernel<<<(int)std::min<int64_t>((words_total + 255) / 256, (int64_t)sm_count * 32), 256, 0, st>>>(
        cube, n_planes, plane_px, n_words, nanbits);
    plane_bits_kernel<<<(n_words + 127) / 128, 128, 0, st>>>(plane_skip, n_planes, n_words, plane_bits);
    count_launches(3);
    return cudaGetLastError();
}

}  // namespace pm
