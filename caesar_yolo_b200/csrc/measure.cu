// Per-source measurements over the catalog boxes (cy_measure_sources / cy_measure_combine, include/caesar_b200.h):
// pixel count, flux sum, peak and weighted first / second moments of the box pixels, read straight from the mosaic
// rows that are already in HBM.
//
// Work is split into units of up to kUnitRows rows of one box, so that a merged hull of thousands of rows spreads over
// many CTAs.  Every unit writes its own partial; the partials of a source are then folded in unit order, and
// cy_measure_combine folds the per-rank arrays in rank order.  Every reduction runs in a fixed order, so the result is
// deterministic for a given row split.
#include "../../include/caesar_b200.h"
#include "common.h"

#include <math.h>
#include <stdint.h>

using namespace cy;

namespace {

constexpr int kUnitRows = 32;     // rows of one box per unit (= per CTA)
constexpr int kThreads = 256;     // 8 warps: warp w reads the unit's rows w, w + 8, ... as coalesced row segments
constexpr int kScanThreads = 1024;

struct Acc {
    long long npix, pidx;
    double peak, sum, sw, swx, swy, swxx, swyy, swxy;
};

__device__ __forceinline__ void acc_init(Acc& a) {
    a.npix = 0;
    a.pidx = LLONG_MAX;
    a.peak = -INFINITY;
    a.sum = a.sw = a.swx = a.swy = a.swxx = a.swyy = a.swxy = 0.0;
}

// peak key (v, -index): larger value wins, lower index on ties
__device__ __forceinline__ void acc_merge(Acc& a, const Acc& b) {
    a.npix += b.npix;
    if (b.peak > a.peak || (b.peak == a.peak && b.pidx < a.pidx)) {
        a.peak = b.peak;
        a.pidx = b.pidx;
    }
    a.sum += b.sum;
    a.sw += b.sw;
    a.swx += b.swx;
    a.swy += b.swy;
    a.swxx += b.swxx;
    a.swyy += b.swyy;
    a.swxy += b.swxy;
}

__device__ __forceinline__ Acc acc_load(const cy_src_partial& p) {
    Acc a;
    a.npix = p.npix;
    a.pidx = p.peak_idx;
    a.peak = p.peak;
    a.sum = p.sum;
    a.sw = p.sw;
    a.swx = p.swx;
    a.swy = p.swy;
    a.swxx = p.swxx;
    a.swyy = p.swyy;
    a.swxy = p.swxy;
    return a;
}

__device__ __forceinline__ void acc_store(cy_src_partial& p, const Acc& a) {
    p.npix = a.npix;
    p.peak_idx = a.pidx;
    p.peak = a.peak;
    p.sum = a.sum;
    p.sw = a.sw;
    p.swx = a.swx;
    p.swy = a.swy;
    p.swxx = a.swxx;
    p.swyy = a.swyy;
    p.swxy = a.swxy;
}

__device__ __forceinline__ Acc acc_shfl_down(const Acc& a, int d) {
    Acc b;
    b.npix = __shfl_down_sync(0xffffffffu, a.npix, d);
    b.pidx = __shfl_down_sync(0xffffffffu, a.pidx, d);
    b.peak = __shfl_down_sync(0xffffffffu, a.peak, d);
    b.sum = __shfl_down_sync(0xffffffffu, a.sum, d);
    b.sw = __shfl_down_sync(0xffffffffu, a.sw, d);
    b.swx = __shfl_down_sync(0xffffffffu, a.swx, d);
    b.swy = __shfl_down_sync(0xffffffffu, a.swy, d);
    b.swxx = __shfl_down_sync(0xffffffffu, a.swxx, d);
    b.swyy = __shfl_down_sync(0xffffffffu, a.swyy, d);
    b.swxy = __shfl_down_sync(0xffffffffu, a.swxy, d);
    return b;
}

// Pixel rectangle of source s inside the owned rows, inclusive bounds; false when empty.  Catalog coordinates are
// integer valued; ceil / floor keep the membership rule x1 <= x <= x2 exact for any value.
struct Box {
    int x0, x1, y0, y1;
};
__device__ __forceinline__ bool source_box(const cy_source& s, int ncols, int row_begin, int row_end, Box& b) {
    const double bx0 = ceil((double)s.x1), bx1 = floor((double)s.x2);
    const double by0 = ceil((double)s.y1), by1 = floor((double)s.y2);
    // the comparisons are false for NaN coordinates
    if (!(bx0 <= bx1 && by0 <= by1 && bx0 <= ncols - 1.0 && bx1 >= 0.0 && by0 <= row_end - 1.0 && by1 >= row_begin))
        return false;
    b.x0 = (int)fmax(bx0, 0.0);
    b.x1 = (int)fmin(bx1, ncols - 1.0);
    b.y0 = (int)fmax(by0, (double)row_begin);
    b.y1 = (int)fmin(by1, row_end - 1.0);
    return b.y0 <= b.y1;   // empty when row_begin == row_end
}

// units per source -> exclusive offsets off[0..nsrc] (one CTA, chunks of kScanThreads sources carried in order)
__global__ void __launch_bounds__(kScanThreads) measure_units_scan_kernel(const cy_source* __restrict__ src, int nsrc,
                                                                           int ncols, int row_begin, int row_end,
                                                                           long long* __restrict__ off) {
    __shared__ long long warp_tot[kScanThreads / 32];
    __shared__ long long carry;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nsrc; base += kScanThreads) {
        const int s = base + t;
        long long c = 0;
        Box b;
        if (s < nsrc && source_box(src[s], ncols, row_begin, row_end, b)) c = (b.y1 - b.y0) / kUnitRows + 1;
        long long inc = c;
        for (int d = 1; d < 32; d <<= 1) {
            const long long v = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += v;
        }
        if (lane == 31) warp_tot[w] = inc;
        __syncthreads();
        long long before = carry;
        for (int k = 0; k < w; ++k) before += warp_tot[k];
        if (s < nsrc) off[s] = before + inc - c;
        __syncthreads();
        if (t == kScanThreads - 1) carry = before + inc;
        __syncthreads();
    }
    if (t == 0) off[nsrc] = carry;
}

// one CTA per unit: partial of up to kUnitRows rows of one box
__global__ void __launch_bounds__(kThreads) measure_unit_kernel(const uint32_t* __restrict__ img, long long row_stride,
                                                                int big_endian, int row0, int ncols,
                                                                const cy_source* __restrict__ src, int nsrc,
                                                                int row_begin, int row_end,
                                                                const long long* __restrict__ off,
                                                                cy_src_partial* __restrict__ unit_out) {
    __shared__ Acc warp_acc[kThreads / 32];
    const long long u = blockIdx.x;
    int lo = 0, hi = nsrc - 1;   // source s with off[s] <= u < off[s + 1] (empty sources share offsets: take the last)
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= u) lo = mid;
        else hi = mid - 1;
    }
    const int s = lo;
    Box b;
    source_box(src[s], ncols, row_begin, row_end, b);
    const int ya = b.y0 + (int)(u - off[s]) * kUnitRows;
    const int yb = min(b.y1, ya + kUnitRows - 1);
    const double cx = ceil((double)src[s].x1), cy = ceil((double)src[s].y1);   // moments about the box corner
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    Acc a;
    acc_init(a);
    for (int y = ya + w; y <= yb; y += kThreads / 32) {
        const uint32_t* row = img + (long long)(y - row0) * row_stride;
        const double dy = (double)y - cy;
        for (int x = b.x0 + lane; x <= b.x1; x += 32) {
            uint32_t raw = __ldg(row + x);
            if (big_endian) raw = __byte_perm(raw, 0, 0x0123);
            const float f = __uint_as_float(raw);
            if (!isfinite(f) || f == 0.0f) continue;   // 0 = masked (utils.py:219,394), non-finite -> masked
            const double v = (double)f;
            const double wgt = fmax(v, 0.0);
            const double dx = (double)x - cx;
            const long long idx = (long long)y * ncols + x;
            a.npix += 1;
            if (v > a.peak) {   // a thread visits its pixels in increasing index order: first hit keeps the tie
                a.peak = v;
                a.pidx = idx;
            }
            a.sum += v;
            a.sw += wgt;
            a.swx += wgt * dx;
            a.swy += wgt * dy;
            a.swxx += wgt * dx * dx;
            a.swyy += wgt * dy * dy;
            a.swxy += wgt * dx * dy;
        }
    }
    for (int d = 16; d > 0; d >>= 1) {
        const Acc o = acc_shfl_down(a, d);
        acc_merge(a, o);
    }
    if (lane == 0) warp_acc[w] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        Acc t = warp_acc[0];
        for (int k = 1; k < kThreads / 32; ++k) acc_merge(t, warp_acc[k]);
        acc_store(unit_out[u], t);
    }
}

// unit partials of each source, folded in unit order -> one partial per source
__global__ void measure_fold_kernel(const cy_src_partial* __restrict__ unit, const long long* __restrict__ off, int nsrc,
                                    cy_src_partial* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsrc) return;
    Acc a;
    acc_init(a);
    for (long long u = off[s]; u < off[s + 1]; ++u) acc_merge(a, acc_load(unit[u]));
    acc_store(out[s], a);
}

__global__ void measure_combine_kernel(const cy_src_partial* __restrict__ part, int world,
                                       const cy_source* __restrict__ src, int nsrc, int ncols,
                                       cy_src_meas* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsrc) return;
    Acc a;
    acc_init(a);
    for (int r = 0; r < world; ++r) acc_merge(a, acc_load(part[(long long)r * nsrc + s]));
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    cy_src_meas m;
    m.npix = a.npix;
    m.sum = a.sum;
    if (a.npix > 0) {
        m.peak = a.peak;
        m.peak_x = (double)(a.pidx % ncols);
        m.peak_y = (double)(a.pidx / ncols);
    } else {
        m.peak = m.peak_x = m.peak_y = nan;
    }
    m.xc = m.yc = m.a = m.b = m.theta = nan;
    if (a.sw > 0.0) {
        const double mx = a.swx / a.sw, my = a.swy / a.sw;   // about the box corner
        m.xc = mx + ceil((double)src[s].x1);
        m.yc = my + ceil((double)src[s].y1);
        const double cxx = fmax(a.swxx / a.sw - mx * mx, 0.0);
        const double cyy = fmax(a.swyy / a.sw - my * my, 0.0);
        const double cxy = a.swxy / a.sw - mx * my;
        const double h = 0.5 * (cxx + cyy), d = sqrt(0.25 * (cxx - cyy) * (cxx - cyy) + cxy * cxy);
        m.a = sqrt(h + d);
        m.b = sqrt(fmax(h - d, 0.0));
        double th = 0.5 * atan2(2.0 * cxy, cxx - cyy) * (180.0 / M_PI);   // (-90, 90]
        if (th <= -90.0) th += 180.0;
        m.theta = th;
    }
    out[s] = m;
}

}  // namespace

extern "C" int cy_measure_sources(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                  const cy_source* src, int nsrc, int row_begin, int row_end, cy_src_partial* partials,
                                  uintptr_t stream) {
    if (nsrc < 0 || ncols <= 0 || row_stride < ncols || row_begin < row0 || row_end < row_begin)
        return set_error(CY_ERR_INVALID, "cy_measure_sources: invalid image geometry or row range");
    if (nsrc == 0) return CY_OK;
    if (!img || !src || !partials) return set_error(CY_ERR_INVALID, "cy_measure_sources: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long* off = nullptr;
    CY_CUDA_CHECK(cudaMallocAsync(&off, (size_t)(nsrc + 1) * sizeof(long long), st));
    measure_units_scan_kernel<<<1, kScanThreads, 0, st>>>(src, nsrc, ncols, row_begin, row_end, off);
    // the unit count is data dependent: bring it to the host
    long long units = 0;
    cudaMemcpyAsync(&units, off + nsrc, sizeof(long long), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        cudaFreeAsync(off, st);
        return set_error(CY_ERR_CUDA, "cy_measure_sources: %s", cudaGetErrorString(e));
    }
    if (units > 2147483647ll) {
        cudaFreeAsync(off, st);
        return set_error(CY_ERR_INVALID, "cy_measure_sources: %lld work units exceed one grid", units);
    }
    cy_src_partial* unit = nullptr;
    if (units > 0 && cudaMallocAsync(&unit, (size_t)units * sizeof(cy_src_partial), st) != cudaSuccess) {
        cudaFreeAsync(off, st);
        return set_error(CY_ERR_NOMEM, "cy_measure_sources: no memory for %lld unit partials", units);
    }
    if (units > 0)
        measure_unit_kernel<<<(unsigned)units, kThreads, 0, st>>>((const uint32_t*)img, row_stride, big_endian, row0,
                                                                  ncols, src, nsrc, row_begin, row_end, off, unit);
    measure_fold_kernel<<<(nsrc + 255) / 256, 256, 0, st>>>(unit, off, nsrc, partials);
    e = cudaGetLastError();
    if (unit) cudaFreeAsync(unit, st);
    cudaFreeAsync(off, st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_measure_sources: %s", cudaGetErrorString(e));
    return CY_OK;
}

extern "C" int cy_measure_combine(const cy_src_partial* partials, int world, const cy_source* src, int nsrc, int ncols,
                                  cy_src_meas* meas, uintptr_t stream) {
    if (world < 1 || nsrc < 0 || ncols <= 0) return set_error(CY_ERR_INVALID, "cy_measure_combine: invalid arguments");
    if (nsrc == 0) return CY_OK;
    if (!partials || !src || !meas) return set_error(CY_ERR_INVALID, "cy_measure_combine: null argument");
    measure_combine_kernel<<<(nsrc + 255) / 256, 256, 0, (cudaStream_t)stream>>>(partials, world, src, nsrc, ncols, meas);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_measure_combine: %s", cudaGetErrorString(e));
    return CY_OK;
}
