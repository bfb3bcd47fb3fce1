// backplane_kernels.cu - fused per-pixel (image direction) and per-cell (map
// direction) backplane kernels, plus the vectorised point transforms.
//
// Work decomposition: one thread per pixel / cell, consecutive threads on consecutive
// elements so every plane store is a fully coalesced 256-byte warp transaction.  A CTA
// of 128 threads stages its frame's constants (PMFrame + values derived once per CTA)
// in shared memory and then processes kPerThread consecutive 128-element segments.
// The grid has one CTA per such chunk (not a persistent grid-stride loop): on-disc
// pixels cost ~10x more than sky pixels, and the hardware CTA scheduler balances that
// dynamically.  __launch_bounds__(128, 4) keeps four CTAs (16 warps) per SM so the
// dependent DFMA chains of neighbouring warps overlap on the FP64 pipe.
// The image kernel is launched as grid (chunks, n_frames): frames of a time series
// are batched into a single launch.
#include "pm_device.cuh"
#include "pm_kernels.h"

#include <cstdlib>

namespace pm {

constexpr int kPerThread = 4;  // elements per thread and CTA (amortises the frame load)
#ifndef PM_IMG_PARAM_CTAS
#define PM_IMG_PARAM_CTAS 4
#endif
constexpr int kImgParamCtas = PM_IMG_PARAM_CTAS;  // resident CTAs per SM the single-frame image kernel is compiled for

// plane slot of id k inside the packed output = number of requested planes below k
__device__ __forceinline__ int slot(uint64_t mask, int k) { return __popcll(mask & (bit(k) - 1ull)); }

// Byte offset of every plane inside the packed plane-major output.  Filled on the host
// and passed BY VALUE as a kernel parameter: parameters live in the constant bank, so a
// store address is `pixel pointer + c[0][offset]` (two integer adds with a constant
// operand) instead of a popcount, a 64-bit multiply and a shared-memory load per store.
struct PlaneOffsets {
    int64_t byte_off[PM_N_PLANES];
    int64_t frame_stride;  // doubles between the plane blocks of consecutive frames
};
static PlaneOffsets make_plane_offsets(uint64_t mask, int64_t plane_stride) {
    PlaneOffsets po;
    int slot = 0;
    for (int k = 0; k < PM_N_PLANES; k++) {
        po.byte_off[k] = (int64_t)slot * plane_stride * (int64_t)sizeof(double);
        if (mask & bit(k)) slot++;
    }
    po.frame_stride = (int64_t)slot * plane_stride;
    return po;
}

// Receives the planes of one pixel / cell and streams them to the plane-major output
struct PlaneSink {
    char *base;  // byte address of this element in plane slot 0
    const PlaneOffsets &po;
    __device__ __forceinline__ void put(int k, double v) const {
        __stcs(reinterpret_cast<double *>(base + po.byte_off[k]), v);
    }
};

// ---------------------------------------------------------------------------------
// Image direction: all requested backplanes for every pixel of every frame.
// ---------------------------------------------------------------------------------
// Pixels idx, idx + 128, ... of this CTA's tile, every requested plane of each
template <bool kSky, uint64_t kFixedMask, bool kSpinSym>
__device__ __forceinline__ void img_tile(const FrameD &fs, uint32_t tile, uint32_t nx, uint32_t npx, int per_thread,
                                         uint64_t mask, const PlaneOffsets &po, double *__restrict__ out) {
    uint32_t idx = tile * (uint32_t)(kBlock * per_thread) + threadIdx.x;
    uint32_t yi = idx / nx, xi = idx - yi * nx;  // one division per thread, then incremental
#pragma unroll 1
    for (int r = 0; r < per_thread && idx < npx; r++) {
        PlaneSink sink{reinterpret_cast<char *>(out + idx), po};
        image_pixel<kSky, kFixedMask, false, kSpinSym>(fs, (double)xi, (double)yi, mask, sink);
        idx += kBlock;
        xi += kBlock;
        while (xi >= nx) {
            xi -= nx;
            yi++;
        }
    }
}

// Batched launch (time series): frame blockIdx.y is staged in shared memory by the CTA.  The frame's
// spin_sym flag is uniform over the CTA, so the branch on it does not diverge.
template <bool kSky, uint64_t kFixedMask>
__global__ void __launch_bounds__(kBlock, 4) backplanes_img_kernel(const PMFrame *__restrict__ frames, uint32_t nx,
                                                                   uint32_t npx, int per_thread, uint64_t mask,
                                                                   const __grid_constant__ PlaneOffsets po,
                                                                   double *__restrict__ out_all) {
    __shared__ FrameD fs;
    load_frame(fs, frames + blockIdx.y);
    double *out = out_all + (int64_t)blockIdx.y * __popcll(mask) * npx;
    if (fs.spin_sym)
        img_tile<kSky, kFixedMask, true>(fs, blockIdx.x, nx, npx, per_thread, mask, po, out);
    else
        img_tile<kSky, kFixedMask, false>(fs, blockIdx.x, nx, npx, per_thread, mask, po, out);
}

// Single frame: the finished constants (derived on the host with the same exactly rounded
// arithmetic as load_frame) arrive as a kernel parameter, i.e. in the constant bank - the FP64
// instructions take them as c[0][offset] operands: no shared-memory loads in the dependency
// chains, no registers holding constants, no CTA prologue and no barrier.
//
// Tiles are handed out from the disc centre outwards (blockIdx.x = 0 is the tile holding the disc
// centre, then alternately the next tile after / before it): CTAs are dispatched in blockIdx order,
// an on-disc tile costs ~10x a sky tile, so the expensive tiles all start first and the kernel
// drains on cheap sky tiles instead of on the last disc rows (longest-processing-time-first).
__device__ __forceinline__ uint32_t centre_out_tile(uint32_t k, uint32_t n_tiles, uint32_t centre) {
    const uint32_t lo = centre, hi = n_tiles - 1u - centre;  // tiles before / after the centre tile
    const uint32_t j = (k + 1u) >> 1;
    if (j <= min(lo, hi)) return (k & 1u) ? centre + j : centre - j;
    return lo < hi ? k : n_tiles - 1u - k;  // one side exhausted: the rest in order, moving away
}
template <bool kSky, uint64_t kFixedMask, bool kSpinSym>
__global__ void __launch_bounds__(kBlock, kImgParamCtas) backplanes_img_param_kernel(
    const __grid_constant__ FrameD fs, uint32_t nx, uint32_t npx, int per_thread, uint32_t centre_tile, uint64_t mask,
    const __grid_constant__ PlaneOffsets po, double *__restrict__ out) {
    img_tile<kSky, kFixedMask, kSpinSym>(fs, centre_out_tile(blockIdx.x, gridDim.x, centre_tile), nx, npx, per_thread,
                                         mask, po, out);
}

// ---------------------------------------------------------------------------------
// Image direction at arbitrary positions (pm_backplanes_points_host): the per-pixel code of the
// single-frame image kernel on a list of (x, y), tiled like map_tile; output plane stride = n
// ---------------------------------------------------------------------------------
template <bool kSky, bool kRingAll, bool kSpinSym>
__global__ void __launch_bounds__(kBlock, 4) backplanes_points_param_kernel(const __grid_constant__ FrameD fs,
                                                                            const double *__restrict__ x_in,
                                                                            const double *__restrict__ y_in,
                                                                            int64_t n, uint64_t mask,
                                                                            const __grid_constant__ PlaneOffsets po,
                                                                            double *__restrict__ out) {
    const int64_t first = (int64_t)blockIdx.x * (kBlock * kPerThread) + threadIdx.x;
#pragma unroll 1
    for (int r = 0; r < kPerThread; r++) {
        const int64_t idx = first + r * kBlock;
        if (idx >= n) break;
        PlaneSink sink{reinterpret_cast<char *>(out + idx), po};
        image_point<kSky, kRingAll, kSpinSym>(fs, __ldg(x_in + idx), __ldg(y_in + idx), mask, sink);
    }
}

// ---------------------------------------------------------------------------------
// Map direction
// ---------------------------------------------------------------------------------
// x_map / y_map of BodyXY.map_img (body_xy.py:3482): the plane set of every reprojection
constexpr uint64_t kXYMapMask = bit(PM_PIXEL_X) | bit(PM_PIXEL_Y);

template <uint64_t kFixedMask>
__device__ __forceinline__ void map_tile(const FrameD &fs, const double *__restrict__ lon_in,
                                         const double *__restrict__ lat_in, int64_t n, uint64_t mask,
                                         const PlaneOffsets &po, double *__restrict__ out) {
    const int64_t first = (int64_t)blockIdx.x * (kBlock * kPerThread) + threadIdx.x;
#pragma unroll 1
    for (int r = 0; r < kPerThread; r++) {
        const int64_t idx = first + r * kBlock;
        if (idx >= n) break;
        PlaneSink sink{reinterpret_cast<char *>(out + idx), po};
        map_cell<kFixedMask>(fs, __ldg(lon_in + idx), __ldg(lat_in + idx), mask, sink);
    }
}

template <uint64_t kFixedMask>
__global__ void __launch_bounds__(kBlock, 4) backplanes_map_kernel(const PMFrame *__restrict__ frame,
                                                                   const double *__restrict__ lon_in,
                                                                   const double *__restrict__ lat_in,
                                                                   int64_t n, uint64_t mask,
                                                                   const __grid_constant__ PlaneOffsets po,
                                                                   double *__restrict__ out) {
    __shared__ FrameD fs;
    // blockIdx.y = frame of a series sharing the lon / lat grid (pm_backplanes_map_batch); each
    // frame's planes follow the previous frame's: po.frame_stride doubles apart
    load_frame(fs, frame + blockIdx.y);
    map_tile<kFixedMask>(fs, lon_in, lat_in, n, mask, po, out + (int64_t)blockIdx.y * po.frame_stride);
}

// Single frame given on the host: constants in the kernel's parameter space, like the image kernel
template <uint64_t kFixedMask>
__global__ void __launch_bounds__(kBlock, 4) backplanes_map_param_kernel(const __grid_constant__ FrameD fs,
                                                                         const double *__restrict__ lon_in,
                                                                         const double *__restrict__ lat_in,
                                                                         int64_t n, uint64_t mask,
                                                                         const __grid_constant__ PlaneOffsets po,
                                                                         double *__restrict__ out) {
    map_tile<kFixedMask>(fs, lon_in, lat_in, n, mask, po, out);
}

// ---------------------------------------------------------------------------------
// Vectorised point transforms.  The per-point loops are shared by the single-frame kernels and their
// time-series counterparts (grid (chunks, n_frames), frame blockIdx.y staged by the CTA, as in
// backplanes_img_kernel): every point of frame f goes through the same device functions with the same
// staged constants, so row f of a batched launch equals the single-frame launch on frame f bit for bit.
// ---------------------------------------------------------------------------------
// Warp-reduced count of missed rays, one atomic per warp that missed
__device__ __forceinline__ void add_missed(unsigned long long missed, unsigned long long *__restrict__ n_missed) {
    for (int o = 16; o > 0; o >>= 1) missed += __shfl_down_sync(0xffffffffu, missed, o);
    if ((threadIdx.x & 31) == 0 && missed) atomicAdd(n_missed, missed);
}

// BodyXY._xy2lonlat (body_xy.py:482-496) -> Body._obsvec_norm2lonlat (body.py:1058-1081)
__device__ __forceinline__ unsigned long long xy2lonlat_tile(const FrameD &fs, const double *__restrict__ xs,
                                                             const double *__restrict__ ys, int64_t n,
                                                             double *__restrict__ lon_out,
                                                             double *__restrict__ lat_out) {
    unsigned long long missed = 0;
    const int64_t first = (int64_t)blockIdx.x * (kBlock * kPerThread) + threadIdx.x;
#pragma unroll 1
    for (int r = 0; r < kPerThread; r++) {
        const int64_t idx = first + r * kBlock;
        if (idx >= n) break;
        const double x = xs[idx], y = ys[idx];
        double lon = NAN, lat = NAN;
        if (fabs(x) < INFINITY && fabs(y) < INFINITY) {
            if (!xy2lonlat_point(fs, x, y, lon, lat)) missed++;
        }
        lon_out[idx] = lon;
        lat_out[idx] = lat;
    }
    return missed;
}
__global__ void __launch_bounds__(kBlock, 4) xy2lonlat_kernel(const PMFrame *__restrict__ frame,
                                                              const double *__restrict__ xs,
                                                              const double *__restrict__ ys, int64_t n,
                                                              double *__restrict__ lon_out,
                                                              double *__restrict__ lat_out,
                                                              unsigned long long *__restrict__ n_missed) {
    __shared__ FrameD fs;
    load_frame(fs, frame);
    const unsigned long long missed = xy2lonlat_tile(fs, xs, ys, n, lon_out, lat_out);
    if (n_missed) add_missed(missed, n_missed);
}
// Time series (pm_xy2lonlat_batch): frame f = blockIdx.y reads its points point_stride doubles after frame
// f - 1's (0: one set shared by every frame), writes row f of the [n_frames][n] outputs, counts into n_missed[f].
// Three CTAs per SM: at four the ray / ellipsoid solve needs more than 128 registers and spills.
__global__ void __launch_bounds__(kBlock, 3) xy2lonlat_batch_kernel(const PMFrame *__restrict__ frames,
                                                                    const double *__restrict__ xs,
                                                                    const double *__restrict__ ys, int64_t n,
                                                                    int64_t point_stride,
                                                                    double *__restrict__ lon_out,
                                                                    double *__restrict__ lat_out,
                                                                    unsigned long long *__restrict__ n_missed) {
    __shared__ FrameD fs;
    load_frame(fs, frames + blockIdx.y);
    const int64_t in = (int64_t)blockIdx.y * point_stride, out = (int64_t)blockIdx.y * n;
    const unsigned long long missed = xy2lonlat_tile(fs, xs + in, ys + in, n, lon_out + out, lat_out + out);
    if (n_missed) add_missed(missed, n_missed + blockIdx.y);
}

// BodyXY._lonlat2xy (body_xy.py:544-560) -> Body._lonlat2obsvec (body.py:1039-1056)
__device__ __forceinline__ void lonlat2xy_tile(const FrameD &fs, const double *__restrict__ lons,
                                               const double *__restrict__ lats, int64_t n, double alt, uint32_t flags,
                                               double *__restrict__ x_out, double *__restrict__ y_out) {
    const int64_t first = (int64_t)blockIdx.x * (kBlock * kPerThread) + threadIdx.x;
#pragma unroll 1
    for (int r = 0; r < kPerThread; r++) {
        const int64_t idx = first + r * kBlock;
        if (idx >= n) break;
        const double lon = lons[idx], lat = lats[idx];
        double x = NAN, y = NAN;
        if (fabs(lon) < INFINITY && fabs(lat) < INFINITY)
            lonlat2xy_point(fs, lon, lat, alt, (flags & PM_FLAG_NOT_VISIBLE_NAN) != 0,
                            (flags & PM_FLAG_PLANETOCENTRIC) != 0, x, y);
        x_out[idx] = x;
        y_out[idx] = y;
    }
}
__global__ void __launch_bounds__(kBlock, 4) lonlat2xy_kernel(const PMFrame *__restrict__ frame,
                                                              const double *__restrict__ lons,
                                                              const double *__restrict__ lats, int64_t n,
                                                              double alt, uint32_t flags,
                                                              double *__restrict__ x_out,
                                                              double *__restrict__ y_out) {
    __shared__ FrameD fs;
    load_frame(fs, frame);
    lonlat2xy_tile(fs, lons, lats, n, alt, flags, x_out, y_out);
}
// Time series (pm_lonlat2xy_batch): layout as xy2lonlat_batch_kernel
__global__ void __launch_bounds__(kBlock, 4) lonlat2xy_batch_kernel(const PMFrame *__restrict__ frames,
                                                                    const double *__restrict__ lons,
                                                                    const double *__restrict__ lats, int64_t n,
                                                                    int64_t point_stride, double alt, uint32_t flags,
                                                                    double *__restrict__ x_out,
                                                                    double *__restrict__ y_out) {
    __shared__ FrameD fs;
    load_frame(fs, frames + blockIdx.y);
    const int64_t in = (int64_t)blockIdx.y * point_stride, out = (int64_t)blockIdx.y * n;
    lonlat2xy_tile(fs, lons + in, lats + in, n, alt, flags, x_out + out, y_out + out);
}

// Generic point transform (pm_transform): any pair of the xy / angular / km / RA-Dec / lon-lat systems.
// Element k < 13 of the frame's default TransformAux: its obsvec -> angular matrix, then the inverse of its
// angular -> km matrix
__device__ __forceinline__ double default_aux(const FrameD &fs, int k) {
    if (k < 9) return fs.f.M[k];
    const double *m = fs.f.ang2km;
    const double det = fma(m[0], m[3], -m[1] * m[2]);
    k -= 9;
    return (k == 0 ? m[3] : k == 1 ? -m[1] : k == 2 ? -m[2] : m[0]) / det;
}
__device__ __forceinline__ unsigned long long transform_tile(const FrameD &fs, const TransformAux &ax, int src, int dst,
                                                             const double *__restrict__ a_in,
                                                             const double *__restrict__ b_in, int64_t n, double alt,
                                                             uint32_t flags, double *__restrict__ a_out,
                                                             double *__restrict__ b_out) {
    unsigned long long missed = 0;
    const int64_t first = (int64_t)blockIdx.x * (kBlock * kPerThread) + threadIdx.x;
#pragma unroll 1
    for (int r = 0; r < kPerThread; r++) {
        const int64_t idx = first + r * kBlock;
        if (idx >= n) break;
        double oa, ob;
        if (!point_transform(fs, ax, src, dst, a_in[idx], b_in[idx], alt, flags, oa, ob)) missed++;
        a_out[idx] = oa;
        b_out[idx] = ob;
    }
    return missed;
}
__global__ void __launch_bounds__(kBlock, 4) transform_kernel(const PMFrame *__restrict__ frame,
                                                              const __grid_constant__ TransformAux aux, int use_aux,
                                                              int src, int dst, const double *__restrict__ a_in,
                                                              const double *__restrict__ b_in, int64_t n, double alt,
                                                              uint32_t flags, double *__restrict__ a_out,
                                                              double *__restrict__ b_out,
                                                              unsigned long long *__restrict__ n_missed) {
    __shared__ FrameD fs;
    __shared__ TransformAux ax;
    load_frame(fs, frame);
    if (threadIdx.x < 13) {
        const double v = !use_aux ? default_aux(fs, threadIdx.x)
                                  : threadIdx.x < 9 ? aux.Mc[threadIdx.x] : aux.km2ang[threadIdx.x - 9];
        (threadIdx.x < 9 ? ax.Mc[threadIdx.x] : ax.km2ang[threadIdx.x - 9]) = v;
    }
    __syncthreads();
    const unsigned long long missed = transform_tile(fs, ax, src, dst, a_in, b_in, n, alt, flags, a_out, b_out);
    if (n_missed) add_missed(missed, n_missed);
}
// Time series (pm_transform_batch): layout as xy2lonlat_batch_kernel; aux13 = [n_frames][13] DEVICE table of
// the frames' TransformAux (row f for frame f), or NULL for every frame's default
__global__ void __launch_bounds__(kBlock, 4) transform_batch_kernel(const PMFrame *__restrict__ frames,
                                                                    const double *__restrict__ aux13, int src,
                                                                    int dst, const double *__restrict__ a_in,
                                                                    const double *__restrict__ b_in, int64_t n,
                                                                    int64_t point_stride, double alt, uint32_t flags,
                                                                    double *__restrict__ a_out,
                                                                    double *__restrict__ b_out,
                                                                    unsigned long long *__restrict__ n_missed) {
    __shared__ FrameD fs;
    __shared__ TransformAux ax;
    load_frame(fs, frames + blockIdx.y);
    if (threadIdx.x < 13) {
        const double v = aux13 ? aux13[(int64_t)blockIdx.y * 13 + threadIdx.x] : default_aux(fs, threadIdx.x);
        (threadIdx.x < 9 ? ax.Mc[threadIdx.x] : ax.km2ang[threadIdx.x - 9]) = v;
    }
    __syncthreads();
    const int64_t in = (int64_t)blockIdx.y * point_stride, out = (int64_t)blockIdx.y * n;
    const unsigned long long missed =
        transform_tile(fs, ax, src, dst, a_in + in, b_in + in, n, alt, flags, a_out + out, b_out + out);
    if (n_missed) add_missed(missed, n_missed + blockIdx.y);
}

// FP64 FMA throughput probes (roofline denominators for the compute-bound kernels): 8 independent
// DFMA chains per thread on a full grid.
//   kind 0: a = fma(a, m, c) with m, c kernel constants - ONE register operand per DFMA.  This is the
//           rate behind the datasheet number (64 FMA / clk / SM).
//   kind 1: a = fma(a, b, d) with three DISTINCT register operands per DFMA - what vector geometry
//           (dot / cross / axpy of per-pixel vectors) issues.  The register file delivers the six
//           32-bit source registers of such an instruction in three cycles, not two, so the pipe
//           sustains 2/3 of the kind-0 rate (tools/microbench/fp64_operands.cu, profiles/r2_summary.md).
template <int kKind>
__global__ void __launch_bounds__(256) fp64_probe_kernel(double *out, const double *in, int iters, double m, double c) {
    double a[8], b[8], d[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        a[i] = threadIdx.x * 1e-9 + i;
        b[i] = kKind ? in[(threadIdx.x + 2 * i + 1) & 63] : m;
        d[i] = kKind ? in[(threadIdx.x + 3 * i + 2) & 63] * 1e-12 : c;
    }
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) a[i] = kKind ? fma(a[i], b[i], d[i]) : fma(a[i], m, c);
    }
    double s = a[0] + a[1] + a[2] + a[3] + a[4] + a[5] + a[6] + a[7];
    if (s == 123.456) out[0] = s;
}

// Device self-test of the pm_math.cuh primitives (tests/test_gpu_math.py):
// kind 0 rcp, 1 rsqrt, 2 sqrt, 3 sin(quarter), 4 cos(quarter), 5 atan2(a, b),
// 6 acos, 7 div(a, b), 8 sin(full), 9 cos(full), 10 atan2(|a|, b), 11 atan2(a, |b|),
// 12 sin, 13 cos of the pixel-offset path (sincos_small2: the tiny-angle tier for |a| <= 2^-8)
__global__ void math_probe_kernel(int kind, const double *__restrict__ a, const double *__restrict__ b,
                                  int64_t n, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double x = a[i], y = b ? b[i] : 0.0;
    double s, c, r = NAN;
    switch (kind) {
        case 0: r = fast_rcp(x); break;
        case 1: r = fast_rsqrt(x); break;
        case 2: r = fast_sqrt(x); break;
        case 3: sincos_small(x, s, c); r = s; break;
        case 4: sincos_small(x, s, c); r = c; break;
        case 5: r = fast_atan2(x, y); break;
        case 6: r = fast_acos(x); break;
        case 7: r = fast_div(x, y); break;
        case 8: sincos_full(x, s, c); r = s; break;
        case 9: sincos_full(x, s, c); r = c; break;
        case 10: r = fast_atan2_ypos(fabs(x), y); break;
        case 11: r = fast_atan2_xpos(x, fabs(y)); break;
        case 12: sincos_small2(x, 0.0, s, c, r, r); r = s; break;
        case 13: sincos_small2(x, 0.0, s, c, r, r); r = c; break;
        default: break;
    }
    out[i] = r;
}

// ---------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------
static unsigned chunks_for(int64_t n) {
    const int64_t per = (int64_t)kBlock * kPerThread;
    int64_t blocks = (n + per - 1) / per;
    return (unsigned)(blocks < 1 ? 1 : blocks);
}

// The default surface stack of BASELINE.json's headline config: lon / lat (graphic + centric),
// incidence / emission / phase, azimuth, local solar time, distance, radial velocity, doppler
constexpr uint64_t kDefaultStackMask = kLonLatMask | kCentricMask | kIllumMask | kStateMask;

// Pixels per thread: as many as possible (amortises the per-CTA frame staging) while the
// grid still has >= 3 waves of resident CTAs for the hardware scheduler to balance.
static int pick_per_thread(int64_t n, int64_t n_batches, int sm_count, int ctas_per_sm) {
    const int64_t tiles = ((n + kBlock - 1) / kBlock) * n_batches;
    const int64_t target = (int64_t)sm_count * ctas_per_sm * 3;
    int per = 16;
    while (per > 1 && tiles / per < target) per >>= 1;
    return per;
}

cudaError_t launch_backplanes_img(const PMFrame *frames, int n_frames, int nx, int ny, uint64_t mask,
                                  double *out, int sm_count, cudaStream_t st) {
    const int64_t npx = (int64_t)nx * ny;
    if (npx >= (1ll << 31)) return cudaErrorInvalidValue;
    const PlaneOffsets po = make_plane_offsets(mask, npx);
    static const int forced = tune_int("PM_IMG_PER_THREAD", 0);
    const int per = forced > 0 ? forced : pick_per_thread(npx, n_frames, sm_count, 4);
    const int64_t chunk = (int64_t)kBlock * per;
    dim3 grid((unsigned)((npx + chunk - 1) / chunk), n_frames);
    static const bool no_fixed = tune_int("PM_IMG_NO_FIXED_MASK", 0) != 0;
    if (mask == kDefaultStackMask && !no_fixed)
        backplanes_img_kernel<false, kDefaultStackMask><<<grid, kBlock, 0, st>>>(frames, (uint32_t)nx, (uint32_t)npx,
                                                                                   per, mask, po, out);
    else if (mask & kSkyMask)
        backplanes_img_kernel<true, 0><<<grid, kBlock, 0, st>>>(frames, (uint32_t)nx, (uint32_t)npx, per, mask, po, out);
    else
        backplanes_img_kernel<false, 0><<<grid, kBlock, 0, st>>>(frames, (uint32_t)nx, (uint32_t)npx, per, mask, po, out);
    count_launches(1);
    return cudaGetLastError();
}
template <bool kSpinSym>
static void launch_img_param(const FrameD &fs, dim3 grid, uint32_t nx, uint32_t npx, int per, uint32_t centre,
                             uint64_t mask, const PlaneOffsets &po, double *out, cudaStream_t st) {
    if (mask == kDefaultStackMask)
        backplanes_img_param_kernel<false, kDefaultStackMask, kSpinSym><<<grid, kBlock, 0, st>>>(fs, nx, npx, per, centre,
                                                                                                mask, po, out);
    else if (mask & kSkyMask)
        backplanes_img_param_kernel<true, 0, kSpinSym><<<grid, kBlock, 0, st>>>(fs, nx, npx, per, centre, mask, po, out);
    else
        backplanes_img_param_kernel<false, 0, kSpinSym><<<grid, kBlock, 0, st>>>(fs, nx, npx, per, centre, mask, po, out);
}
// single frame given on the HOST: constants derived here, passed by value; the frame's spin_sym flag
// picks the instantiation, so each kernel carries one path's code and registers only
cudaError_t launch_backplanes_img_host(const PMFrame *frame_host, int nx, int ny, uint64_t mask, double *out,
                                       int sm_count, cudaStream_t st) {
    const int64_t npx = (int64_t)nx * ny;
    if (npx >= (1ll << 31)) return cudaErrorInvalidValue;
    FrameD fs;
    load_frame_host(fs, frame_host);
    const PlaneOffsets po = make_plane_offsets(mask, npx);
    static const int forced = tune_int("PM_IMG_PER_THREAD", 0);
    const int per = forced > 0 ? forced : pick_per_thread(npx, 1, sm_count, kImgParamCtas);
    const int64_t chunk = (int64_t)kBlock * per;
    const int64_t n_tiles = (npx + chunk - 1) / chunk;
    dim3 grid((unsigned)n_tiles, 1);
    // tile of the disc centre (clamped into the frame); tune: PM_IMG_ORDER=0 keeps the linear order
    double cy = frame_host->y0 < 0.0 ? 0.0 : (frame_host->y0 > ny - 1.0 ? ny - 1.0 : frame_host->y0);
    double cx = frame_host->x0 < 0.0 ? 0.0 : (frame_host->x0 > nx - 1.0 ? nx - 1.0 : frame_host->x0);
    if (!(cy == cy) || !(cx == cx)) cy = cx = 0.0;
    int64_t ct = ((int64_t)cy * nx + (int64_t)cx) / chunk;
    static const bool linear = tune_int("PM_IMG_ORDER", 1) == 0;
    if (linear) ct = 0;
    const uint32_t centre = (uint32_t)(ct < 0 ? 0 : (ct >= n_tiles ? n_tiles - 1 : ct));
    if (fs.spin_sym)
        launch_img_param<true>(fs, grid, (uint32_t)nx, (uint32_t)npx, per, centre, mask, po, out, st);
    else
        launch_img_param<false>(fs, grid, (uint32_t)nx, (uint32_t)npx, per, centre, mask, po, out, st);
    count_launches(1);
    return cudaGetLastError();
}
template <bool kSpinSym>
static void launch_points_param(const FrameD &fs, unsigned grid, const double *x, const double *y, int64_t n,
                                uint64_t mask, uint32_t flags, const PlaneOffsets &po, double *out, cudaStream_t st) {
    // the ring planes are sky planes: without a sky plane PM_FLAG_RING_ALL has nothing to change
    if (!(mask & kSkyMask))
        backplanes_points_param_kernel<false, false, kSpinSym><<<grid, kBlock, 0, st>>>(fs, x, y, n, mask, po, out);
    else if (flags & PM_FLAG_RING_ALL)
        backplanes_points_param_kernel<true, true, kSpinSym><<<grid, kBlock, 0, st>>>(fs, x, y, n, mask, po, out);
    else
        backplanes_points_param_kernel<true, false, kSpinSym><<<grid, kBlock, 0, st>>>(fs, x, y, n, mask, po, out);
}
// n arbitrary image positions of ONE frame given on the HOST (constants derived here, as above)
cudaError_t launch_backplanes_points_host(const PMFrame *frame_host, const double *x, const double *y, int64_t n,
                                          uint64_t mask, uint32_t flags, double *out, cudaStream_t st) {
    FrameD fs;
    load_frame_host(fs, frame_host);
    const PlaneOffsets po = make_plane_offsets(mask, n);
    const unsigned grid = chunks_for(n);
    if (fs.spin_sym)
        launch_points_param<true>(fs, grid, x, y, n, mask, flags, po, out, st);
    else
        launch_points_param<false>(fs, grid, x, y, n, mask, flags, po, out, st);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_backplanes_map(const PMFrame *frames, int n_frames, const double *lon, const double *lat,
                                  int64_t n, uint64_t mask, double *out, int sm_count, cudaStream_t st) {
    (void)sm_count;
    const dim3 grid(chunks_for(n), (unsigned)n_frames);
    const PlaneOffsets po = make_plane_offsets(mask, n);
    if (mask == kXYMapMask)
        backplanes_map_kernel<kXYMapMask><<<grid, kBlock, 0, st>>>(frames, lon, lat, n, mask, po, out);
    else
        backplanes_map_kernel<0><<<grid, kBlock, 0, st>>>(frames, lon, lat, n, mask, po, out);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_backplanes_map_host(const PMFrame *frame_host, const double *lon, const double *lat, int64_t n,
                                       uint64_t mask, double *out, int sm_count, cudaStream_t st) {
    (void)sm_count;
    FrameD fs;
    load_frame_host(fs, frame_host);
    const PlaneOffsets po = make_plane_offsets(mask, n);
    if (mask == kXYMapMask)
        backplanes_map_param_kernel<kXYMapMask><<<chunks_for(n), kBlock, 0, st>>>(fs, lon, lat, n, mask, po, out);
    else
        backplanes_map_param_kernel<0><<<chunks_for(n), kBlock, 0, st>>>(fs, lon, lat, n, mask, po, out);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_xy2lonlat(const PMFrame *frame, const double *x, const double *y, int64_t n, double *lon,
                             double *lat, unsigned long long *n_missed, int sm_count, cudaStream_t st) {
    (void)sm_count;
    xy2lonlat_kernel<<<chunks_for(n), kBlock, 0, st>>>(frame, x, y, n, lon, lat, n_missed);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_lonlat2xy(const PMFrame *frame, const double *lon, const double *lat, int64_t n, double alt,
                             uint32_t flags, double *x, double *y, int sm_count, cudaStream_t st) {
    (void)sm_count;
    lonlat2xy_kernel<<<chunks_for(n), kBlock, 0, st>>>(frame, lon, lat, n, alt, flags, x, y);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_transform(const PMFrame *frame, int src, int dst, const double *a, const double *b, int64_t n,
                             double alt, uint32_t flags, const double *aux13_host, double *out_a, double *out_b,
                             unsigned long long *n_missed, cudaStream_t st) {
    TransformAux aux = {};
    if (aux13_host) {
        for (int i = 0; i < 9; i++) aux.Mc[i] = aux13_host[i];
        for (int i = 0; i < 4; i++) aux.km2ang[i] = aux13_host[9 + i];
    }
    transform_kernel<<<chunks_for(n), kBlock, 0, st>>>(frame, aux, aux13_host != nullptr, src, dst, a, b, n, alt,
                                                       flags, out_a, out_b, n_missed);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_xy2lonlat_batch(const PMFrame *frames, int n_frames, const double *x, const double *y, int64_t n,
                                   int64_t point_stride, double *lon, double *lat, unsigned long long *n_missed,
                                   cudaStream_t st) {
    xy2lonlat_batch_kernel<<<dim3(chunks_for(n), (unsigned)n_frames), kBlock, 0, st>>>(frames, x, y, n, point_stride,
                                                                                       lon, lat, n_missed);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_lonlat2xy_batch(const PMFrame *frames, int n_frames, const double *lon, const double *lat,
                                   int64_t n, int64_t point_stride, double alt, uint32_t flags, double *x, double *y,
                                   cudaStream_t st) {
    lonlat2xy_batch_kernel<<<dim3(chunks_for(n), (unsigned)n_frames), kBlock, 0, st>>>(frames, lon, lat, n,
                                                                                       point_stride, alt, flags, x, y);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_transform_batch(const PMFrame *frames, int n_frames, int src, int dst, const double *a,
                                   const double *b, int64_t n, int64_t point_stride, double alt, uint32_t flags,
                                   const double *aux13, double *out_a, double *out_b, unsigned long long *n_missed,
                                   cudaStream_t st) {
    transform_batch_kernel<<<dim3(chunks_for(n), (unsigned)n_frames), kBlock, 0, st>>>(
        frames, aux13, src, dst, a, b, n, point_stride, alt, flags, out_a, out_b, n_missed);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_fp64_probe(double *scratch, int kind, int iters, int sm_count, cudaStream_t st) {
    // scratch: >= 65 doubles; [1 .. 64] hold values near 1 (filled by the caller), [0] is the sink
    if (kind == 0)
        fp64_probe_kernel<0><<<sm_count * 8, 256, 0, st>>>(scratch, scratch + 1, iters, 0.999999999, 1e-12);
    else
        fp64_probe_kernel<1><<<sm_count * 8, 256, 0, st>>>(scratch, scratch + 1, iters, 0.999999999, 1e-12);
    count_launches(1);
    return cudaGetLastError();
}
cudaError_t launch_math_probe(int kind, const double *a, const double *b, int64_t n, double *out,
                              cudaStream_t st) {
    math_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(kind, a, b, n, out);
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace pm
