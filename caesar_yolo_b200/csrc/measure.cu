// Per-source measurements over the catalog boxes (cy_measure_sources / cy_measure_combine, include/caesar_b200.h):
// pixel count, flux sum, peak and weighted first / second moments of the box pixels, read straight from the mosaic
// rows that are already in HBM.  The local background and noise (cy_noise_init / cy_noise_pass / cy_noise_update) take
// the sigma-clipped mean and standard deviation of a frame around each box from the same rows, one pass per clip.
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

// Pixel rectangle of source s grown by `grow` pixels on every side (0: the box itself; the noise frame's outer edge),
// inside the image columns and the owned rows, inclusive bounds; false when empty or when the box itself is empty.
// Catalog coordinates are integer valued; ceil / floor keep the membership rule x1 <= x <= x2 exact for any value.
struct Box {
    int x0, x1, y0, y1;
};
__device__ __forceinline__ bool source_box(const cy_source& s, int grow, int ncols, int row_begin, int row_end, Box& b) {
    const double bx0 = ceil((double)s.x1), bx1 = floor((double)s.x2);
    const double by0 = ceil((double)s.y1), by1 = floor((double)s.y2);
    // the comparisons are false for NaN coordinates
    if (!(bx0 <= bx1 && by0 <= by1)) return false;
    const double gx0 = bx0 - grow, gx1 = bx1 + grow, gy0 = by0 - grow, gy1 = by1 + grow;
    if (!(gx0 <= ncols - 1.0 && gx1 >= 0.0 && gy0 <= row_end - 1.0 && gy1 >= row_begin)) return false;
    b.x0 = (int)fmax(gx0, 0.0);
    b.x1 = (int)fmin(gx1, ncols - 1.0);
    b.y0 = (int)fmax(gy0, (double)row_begin);
    b.y1 = (int)fmin(gy1, row_end - 1.0);
    return b.y0 <= b.y1;   // empty when row_begin == row_end
}

// source of work unit u: s with off[s] <= u < off[s + 1] (empty sources share offsets: take the last)
__device__ __forceinline__ int unit_source(const long long* __restrict__ off, int nsrc, long long u) {
    int lo = 0, hi = nsrc - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= u) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// units of items 0..n-1 (count(s)) -> exclusive offsets off[0..n] (one CTA of kScanThreads threads, chunks of
// kScanThreads items carried in order)
template <typename Count>
__device__ __forceinline__ void scan_units(int nsrc, Count count, long long* __restrict__ off) {
    __shared__ long long warp_tot[kScanThreads / 32];
    __shared__ long long carry;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nsrc; base += kScanThreads) {
        const int s = base + t;
        const long long c = s < nsrc ? count(s) : 0;
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

struct SourceUnits {
    const cy_source* src;
    int grow, ncols, row_begin, row_end;
    __device__ long long operator()(int s) const {
        Box b;
        return source_box(src[s], grow, ncols, row_begin, row_end, b) ? (b.y1 - b.y0) / kUnitRows + 1 : 0;
    }
};

// units per source (rows of the box grown by `grow`) -> exclusive offsets off[0..nsrc]
__global__ void __launch_bounds__(kScanThreads) measure_units_scan_kernel(const cy_source* __restrict__ src, int nsrc,
                                                                           int grow, int ncols, int row_begin,
                                                                           int row_end, long long* __restrict__ off) {
    scan_units(nsrc, SourceUnits{src, grow, ncols, row_begin, row_end}, off);
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
    const int s = unit_source(off, nsrc, u);
    Box b;
    source_box(src[s], 0, ncols, row_begin, row_end, b);
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

// ---------------------------------------------------------------------------------------------- frame noise
// One pass of the iterative sigma clipping of every active source's frame (cy_noise_pass / cy_noise_update): the units
// are the rows of the grown box (measure_units_scan_kernel with grow = frame), scanned once per measurement.

constexpr double kClipSigma = 3.0;   // kappa
constexpr int kClipMaxIters = 5;     // passes 0..5: the statistics of all pixels, then up to 5 clipped sets

struct NAcc {
    long long n;
    double s1, s2;
};

__device__ __forceinline__ void nacc_merge(NAcc& a, const NAcc& b) {
    a.n += b.n;
    a.s1 += b.s1;
    a.s2 += b.s2;
}

// decoded pixel value, NaN when masked: non-finite pixels and 0 (the masking rule of the box measurements)
__device__ __forceinline__ float noise_pixel(const uint32_t* p, int big_endian) {
    uint32_t raw = __ldg(p);
    if (big_endian) raw = __byte_perm(raw, 0, 0x0123);
    const float f = __uint_as_float(raw);
    return (isfinite(f) && f != 0.0f) ? f : __int_as_float(0x7fc00000);
}

// ---- median select (cy_noise_pass_median, cy_bkg_grid_pass_median, cy_median_update).  A kept pixel's key is the
// order-preserving map of its float32 bits (negative: all bits flipped; positive: sign bit set; 0 and non-finite values
// are masked).  Round r counts byte r (from the top) of the keys whose top 8r bits equal the prefix of a middle rank:
// slots [0, 256) for the lower middle rank, [256, 512) for the upper one once their prefixes differ.
constexpr int kSelectBins = 256;
constexpr int kSelectSlots = 2 * kSelectBins;
constexpr int kSelectRounds = 4;

__device__ __forceinline__ uint32_t float_key(uint32_t bits) {
    return (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
}

__device__ __forceinline__ uint32_t key_bits(uint32_t key) {
    return (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
}

struct Select {
    uint32_t p0, p1;
    int round, split, shift;   // shift = 32 - 8 round: the prefix of a key is key >> shift (round >= 1)
};

__device__ __forceinline__ Select select_load(const cy_select_state& t, int round) {
    return Select{t.prefix[0], t.prefix[1], round, round > 0 ? t.split : 0, 32 - 8 * round};
}

// the kept pixel with float bits `bits` -> its slot, counted once per distinct slot of the warp (all 32 lanes call)
__device__ __forceinline__ void select_count(uint32_t* h, const Select& q, bool keep, uint32_t bits) {
    int slot = -1;
    if (keep) {
        const uint32_t key = float_key(bits);
        if (q.round == 0) {
            slot = (int)(key >> 24);
        } else {
            const uint32_t pre = key >> q.shift, b = (key >> (q.shift - 8)) & 255u;
            if (pre == q.p0) slot = (int)b;
            else if (q.split && pre == q.p1) slot = kSelectBins + (int)b;
        }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, slot);
    if (slot >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(h + slot, (uint32_t)__popc(peers));
}

// shared slots -> the global histogram of the source or node (integer adds: any order gives the same counts)
__device__ __forceinline__ void select_flush(const uint32_t* h, uint32_t* __restrict__ out, int t, int nt) {
    for (int i = t; i < kSelectSlots; i += nt)
        if (h[i]) atomicAdd(out + i, h[i]);
}

__global__ void noise_init_kernel(int nsrc, cy_noise_state* __restrict__ state) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsrc) return;
    cy_noise_state t;
    t.lo = -INFINITY;
    t.hi = INFINITY;
    t.c = 0.0;
    t.bkg = t.rms = __longlong_as_double(0x7ff8000000000000ll);
    t.nbkg = 0;
    t.iters = 0;
    t.done = 0;
    state[s] = t;
}

// one CTA per unit: sums of (v - c), (v - c)^2 over the frame pixels of up to kUnitRows rows of one grown box that lie
// inside the source's kept interval [lo, hi].  Rows inside the box's row span read the two side segments, packed into
// one run of lane indices; other rows read the full grown width.  A converged source's units return at once.
// kMask: a pixel whose bit is set in the source mask (cy_source_mask over the same ncols and rows) is skipped before
// its load; the unmasked instantiation does not touch `mask`.
// kMedian: one digit round of the median select (select_count): round 0 also sums the moments, rounds 1..3 only count;
// the CTA's histogram goes to hist[s * kSelectSlots ..] with integer atomics.  The mean instantiation does not touch
// sel, round or hist.
template <bool kMask, bool kMedian = false>
__global__ void __launch_bounds__(kThreads) noise_unit_kernel(const uint32_t* __restrict__ img, long long row_stride,
                                                              int big_endian, int row0, int ncols,
                                                              const cy_source* __restrict__ src, int nsrc,
                                                              int row_begin, int row_end, int frame,
                                                              const long long* __restrict__ off,
                                                              const cy_noise_state* __restrict__ state,
                                                              cy_noise_partial* __restrict__ unit_out,
                                                              const uint32_t* __restrict__ mask,
                                                              const cy_select_state* __restrict__ sel = nullptr,
                                                              int round = 0, uint32_t* __restrict__ hist = nullptr) {
    __shared__ NAcc warp_acc[kThreads / 32];
    const long long u = blockIdx.x;
    const int s = unit_source(off, nsrc, u);
    if (state[s].done) return;
    const double lo = state[s].lo, hi = state[s].hi, c = state[s].c;
    Box g;
    source_box(src[s], frame, ncols, row_begin, row_end, g);
    const double bx0 = ceil((double)src[s].x1), bx1 = floor((double)src[s].x2);
    const double by0 = ceil((double)src[s].y1), by1 = floor((double)src[s].y2);
    // side segments of a box row: [g.x0, g.x0 + nl) and [r0, r0 + nr), both inside [g.x0, g.x1]
    const int l1 = (int)fmax(fmin(bx0 - 1.0, (double)g.x1), g.x0 - 1.0);
    const int r0 = (int)fmin(fmax(bx1 + 1.0, (double)g.x0), g.x1 + 1.0);
    const int side_l = l1 - g.x0 + 1, side_r = g.x1 - r0 + 1;
    const int ya = g.y0 + (int)(u - off[s]) * kUnitRows;
    const int yb = min(g.y1, ya + kUnitRows - 1);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    NAcc a = {0, 0.0, 0.0};
    if constexpr (kMedian) {
        __shared__ uint32_t s_hist[kSelectSlots];
        for (int i = threadIdx.x; i < kSelectSlots; i += kThreads) s_hist[i] = 0;
        __syncthreads();
        const Select q = select_load(sel[s], round);
        for (int y = ya + w; y <= yb; y += kThreads / 32) {
            const uint32_t* row = img + (long long)(y - row0) * row_stride;
            const uint32_t* mrow = kMask ? mask + (long long)(y - row_begin) * ((ncols + 31) >> 5) : nullptr;
            const bool in_box = (double)y >= by0 && (double)y <= by1;
            const int nl = in_box ? side_l : g.x1 - g.x0 + 1, nr = in_box ? side_r : 0;
            for (int i0 = 0; i0 < nl + nr; i0 += 32) {   // the warp stays converged for select_count
                const int i = i0 + lane, x = i < nl ? g.x0 + i : r0 + (i - nl);
                float f = __int_as_float(0x7fc00000);
                if (i < nl + nr && !(kMask && ((__ldg(mrow + (x >> 5)) >> (x & 31)) & 1u)))
                    f = noise_pixel(row + x, big_endian);
                const double v = (double)f;
                const bool keep = v >= lo && v <= hi;   // false for a masked pixel (NaN)
                if (keep && round == 0) {
                    const double d = v - c;
                    a.n += 1;
                    a.s1 += d;
                    a.s2 += d * d;
                }
                select_count(s_hist, q, keep, __float_as_uint(f));
            }
        }
        __syncthreads();
        select_flush(s_hist, hist + (long long)s * kSelectSlots, threadIdx.x, kThreads);
        if (round != 0) return;
    } else {
        for (int y = ya + w; y <= yb; y += kThreads / 32) {
            const uint32_t* row = img + (long long)(y - row0) * row_stride;
            const uint32_t* mrow = kMask ? mask + (long long)(y - row_begin) * ((ncols + 31) >> 5) : nullptr;
            const bool in_box = (double)y >= by0 && (double)y <= by1;
            const int nl = in_box ? side_l : g.x1 - g.x0 + 1, nr = in_box ? side_r : 0;
            for (int i = lane; i < nl + nr; i += 32) {
                const int x = i < nl ? g.x0 + i : r0 + (i - nl);
                if (kMask && ((__ldg(mrow + (x >> 5)) >> (x & 31)) & 1u)) continue;
                const double v = (double)noise_pixel(row + x, big_endian);
                if (!(v >= lo && v <= hi)) continue;       // false for a masked pixel (NaN)
                const double d = v - c;
                a.n += 1;
                a.s1 += d;
                a.s2 += d * d;
            }
        }
    }
    for (int d = 16; d > 0; d >>= 1) {
        NAcc o;
        o.n = __shfl_down_sync(0xffffffffu, a.n, d);
        o.s1 = __shfl_down_sync(0xffffffffu, a.s1, d);
        o.s2 = __shfl_down_sync(0xffffffffu, a.s2, d);
        nacc_merge(a, o);
    }
    if (lane == 0) warp_acc[w] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        NAcc t = warp_acc[0];
        for (int k = 1; k < kThreads / 32; ++k) nacc_merge(t, warp_acc[k]);
        unit_out[u].n = t.n;
        unit_out[u].s1 = t.s1;
        unit_out[u].s2 = t.s2;
    }
}

// unit partials of each active source, folded in unit order -> one partial per source (zero without units)
__global__ void noise_fold_kernel(const cy_noise_partial* __restrict__ unit, const long long* __restrict__ off,
                                  int nsrc, const cy_noise_state* __restrict__ state,
                                  cy_noise_partial* __restrict__ out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsrc || state[s].done) return;
    NAcc a = {0, 0.0, 0.0};
    for (long long u = off[s]; u < off[s + 1]; ++u) {
        const NAcc b = {unit[u].n, unit[u].s1, unit[u].s2};
        nacc_merge(a, b);
    }
    out[s].n = a.n;
    out[s].s1 = a.s1;
    out[s].s2 = a.s2;
}

// partials [world][nsrc] folded in rank order -> statistics of the pass just run; either the source stops (final bkg,
// rms, nbkg, iters) or its interval, shift and pass index advance.  *active counts the sources that go on.
__global__ void noise_update_kernel(const cy_noise_partial* __restrict__ part, int world, int nsrc,
                                    cy_noise_state* __restrict__ state, int* __restrict__ active) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsrc) return;
    cy_noise_state t = state[s];
    if (t.done) return;
    NAcc a = {0, 0.0, 0.0};
    for (int r = 0; r < world; ++r) {
        const cy_noise_partial& p = part[(long long)r * nsrc + s];
        const NAcc b = {p.n, p.s1, p.s2};
        nacc_merge(a, b);
    }
    const int k = t.iters;   // index of the pass just run
    if (a.n == 0) {          // empty frame (a clipped set is never empty: it holds the pixels within sigma of the mean)
        t.nbkg = 0;
        t.bkg = t.rms = __longlong_as_double(0x7ff8000000000000ll);
        t.done = 1;
        state[s] = t;
        return;
    }
    const double m1 = a.s1 / (double)a.n;
    const double mu = t.c + m1;
    const double sd = sqrt(fmax(a.s2 / (double)a.n - m1 * m1, 0.0));
    t.bkg = mu;
    t.rms = sd;
    if ((k >= 1 && a.n == t.nbkg) || k == kClipMaxIters) {
        t.done = 1;
    } else {
        t.lo = fmax(t.lo, mu - kClipSigma * sd);
        t.hi = fmin(t.hi, mu + kClipSigma * sd);
        t.c = mu;
        t.iters = k + 1;
        atomicAdd(active, 1);
    }
    t.nbkg = a.n;
    state[s] = t;
}

// Walks the bins of one digit: the bin that holds rank `rank` (0-based) of the counted keys; rank becomes the rank
// inside that bin and the bin is appended to the prefix.
__device__ __forceinline__ void select_pick(const uint32_t* __restrict__ h, int64_t& rank, uint32_t& prefix) {
    int b = 0;
    long long below = 0;
    for (; b < kSelectBins - 1; ++b) {
        const long long c = h[b];
        if (rank < below + c) break;
        below += c;
    }
    rank -= below;
    prefix = (prefix << 8) | (uint32_t)b;
}

// Round `round` of pass k, after the histograms of every rank are summed.  Round 0 also folds the moment partials
// [world][n] in rank order (as noise_update_kernel): an empty set or n_k = n_{k-1} stops the source here (the set did
// not change, so its median is the shift c = m_{k-1}); otherwise the middle ranks of the n_k kept pixels are set.
// Every round picks the bins of both ranks; round 3 has their full keys, finalises m_k and advances the state like
// noise_update_kernel with the median as the centre.  cnt[0] counts the sources that go on, cnt[1] the sets of
// 2^32 pixels or more (their uint32 bins can wrap).
__global__ void median_update_kernel(const cy_noise_partial* __restrict__ part, int world,
                                     const uint32_t* __restrict__ hist, int nsrc, cy_noise_state* __restrict__ state,
                                     cy_select_state* __restrict__ sel, int round, int* __restrict__ cnt) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nsrc) return;
    cy_noise_state t = state[s];
    if (t.done) return;
    cy_select_state q = sel[s];
    const int k = t.iters;   // index of the pass
    if (round == 0) {
        NAcc a = {0, 0.0, 0.0};
        for (int r = 0; r < world; ++r) {
            const cy_noise_partial& p = part[(long long)r * nsrc + s];
            const NAcc b = {p.n, p.s1, p.s2};
            nacc_merge(a, b);
        }
        if (a.n == 0) {
            t.nbkg = 0;
            t.bkg = t.rms = __longlong_as_double(0x7ff8000000000000ll);
            t.done = 1;
            state[s] = t;
            return;
        }
        const double m1 = a.s1 / (double)a.n;
        t.rms = sqrt(fmax(a.s2 / (double)a.n - m1 * m1, 0.0));
        if (k >= 1 && a.n == t.nbkg) {
            t.bkg = t.c;
            t.done = 1;
            state[s] = t;
            return;
        }
        state[s] = t;
        q.n = a.n;
        q.rank[0] = (a.n - 1) / 2;   // x_((n-1)/2) and x_(n/2): the same rank for odd n
        q.rank[1] = a.n / 2;
        q.prefix[0] = q.prefix[1] = 0;
        q.split = 0;
    }
    const uint32_t* h = hist + (long long)s * kSelectSlots;
    select_pick(h, q.rank[0], q.prefix[0]);
    select_pick(q.split ? h + kSelectBins : h, q.rank[1], q.prefix[1]);
    q.split = q.prefix[0] != q.prefix[1];
    q.round = round;
    sel[s] = q;
    if (round < kSelectRounds - 1) return;
    if (q.n > 0xffffffffll) atomicAdd(cnt + 1, 1);
    const double m = ((double)__uint_as_float(key_bits(q.prefix[0])) +
                      (double)__uint_as_float(key_bits(q.prefix[1]))) / 2.0;   // np.median of the fp64 values
    const double sd = t.rms;
    t.bkg = m;
    if (k == kClipMaxIters) {
        t.done = 1;
    } else {
        t.lo = fmax(t.lo, m - kClipSigma * sd);
        t.hi = fmin(t.hi, m + kClipSigma * sd);
        t.c = m;
        t.iters = k + 1;
        atomicAdd(cnt, 1);
    }
    t.nbkg = q.n;
    state[s] = t;
}

// ---------------------------------------------------------------------------------------------- background maps
// The sigma clipping above over the boxes of a node lattice (cy_bkg_grid_init / cy_bkg_grid_pass / cy_bkg_grid_maps).
// A work unit is one chunk of <= kUnitRows rows of one node row and a group of kGridNodes adjacent node columns: the CTA
// copies the columns its active nodes cover into shared memory once per chunk, slice by slice, and every warp folds
// them into its nodes' sums.  Node rows overlap vertically (box / grid ~ 4 at the defaults); that re-read stays.

constexpr int kGridNodes = 16;                          // node columns per unit: warp w takes nodes w and w + 8
constexpr int kNodesPerWarp = kGridNodes / (kThreads / 32);
constexpr int kSliceCols = 256;                         // columns of one shared-memory slice (32 KB with kUnitRows)
constexpr int kBkgSelectSmem = (kGridNodes * kSelectSlots + 3 * kGridNodes) * 4;   // median select: 32.2 KB

// Node lattice of the region: columns [0, ncols) of the buffer, rows [R0, R1); rlo..rhi: the rows of this range
// (inclusive; empty when rlo > rhi).  h is clipped to the region's larger side, which changes no box.
struct Grid {
    int ncols, R0, R1, g, h, nx, ny, ngroups, rlo, rhi;
    __host__ __device__ int xnode(int i) const { return (int)min((long long)i * g, (long long)ncols - 1); }
    __host__ __device__ int ynode(int j) const { return R0 + (int)min((long long)j * g, (long long)(R1 - R0) - 1); }
    // rows of node row j inside this range, inclusive; false when none
    __host__ __device__ bool rows(int j, int& a, int& b) const {
        a = max(ynode(j) - h, rlo);
        b = min(ynode(j) + h, rhi);
        return a <= b;
    }
};

static bool make_grid(int ncols, int R0, int R1, int row_begin, int row_end, int box, int grid, Grid& G) {
    if (ncols < 1 || R1 <= R0 || row_begin < R0 || row_end < row_begin || row_end > R1 || box < 3 || !(box & 1) ||
        grid < 1)
        return false;
    const int H = R1 - R0;
    G.ncols = ncols;
    G.R0 = R0;
    G.R1 = R1;
    G.g = grid;
    G.h = min(box / 2, max(ncols, H));
    G.nx = (int)(((long long)ncols - 1 + grid - 1) / grid) + 1;
    G.ny = (int)(((long long)H - 1 + grid - 1) / grid) + 1;
    G.ngroups = (G.nx + kGridNodes - 1) / kGridNodes;
    G.rlo = row_begin;
    G.rhi = row_end - 1;
    return (long long)G.nx * G.ny <= 2147483647ll;
}

struct NodeRowUnits {
    Grid G;
    __device__ long long operator()(int j) const {
        int a, b;
        return G.rows(j, a, b) ? (long long)((b - a) / kUnitRows + 1) * G.ngroups : 0;
    }
};

__global__ void __launch_bounds__(kScanThreads) bkg_units_scan_kernel(Grid G, long long* __restrict__ off) {
    scan_units(G.ny, NodeRowUnits{G}, off);
}

// one CTA per unit: sums of (v - c), (v - c)^2 over the pixels of the unit's rows inside each active node's box and
// kept interval -> unit_out[u * kGridNodes + k] for node column i0 + k.  A unit whose nodes are all done returns at once;
// only the columns from the first to the last active node's box are read.
// kMask: region pixel (x, y) is masked when bit x + mask_col0 of mask row y - G.rlo is set (mask_words words per row);
// it enters the shared tile as NaN, so the fold loop is that of the unmasked instantiation, which does not touch `mask`.
// kMedian: one digit round of the median select, as for noise_unit_kernel; the kGridNodes histograms and the nodes'
// prefixes live in kBkgSelectSmem bytes of dynamic shared memory, and a node's slots go to hist[n * kSelectSlots ..].
template <bool kMask, bool kMedian = false>
__global__ void __launch_bounds__(kThreads) bkg_unit_kernel(const uint32_t* __restrict__ img, long long row_stride,
                                                            int big_endian, int row0, Grid G,
                                                            const long long* __restrict__ off,
                                                            const cy_noise_state* __restrict__ state,
                                                            cy_noise_partial* __restrict__ unit_out,
                                                            const uint32_t* __restrict__ mask, int mask_words,
                                                            int mask_col0,
                                                            const cy_select_state* __restrict__ sel = nullptr,
                                                            int round = 0, uint32_t* __restrict__ hist = nullptr) {
    __shared__ float tile[kUnitRows][kSliceCols];
    __shared__ double s_lo[kGridNodes], s_hi[kGridNodes], s_c[kGridNodes];
    __shared__ int s_active[kGridNodes];
    const long long u = blockIdx.x;
    const int j = unit_source(off, G.ny, u);
    const long long local = u - off[j];
    const int grp = (int)(local % G.ngroups), chunk = (int)(local / G.ngroups);
    const int i0 = grp * kGridNodes, ni = min(kGridNodes, G.nx - i0);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x < kGridNodes) {
        const int k = threadIdx.x;
        int act = 0;
        if (k < ni) {
            const cy_noise_state& s = state[(long long)j * G.nx + i0 + k];
            act = !s.done;
            s_lo[k] = s.lo;
            s_hi[k] = s.hi;
            s_c[k] = s.c;
        }
        s_active[k] = act;
    }
    if constexpr (kMedian) {
        extern __shared__ uint32_t s_sel[];   // [kGridNodes][kSelectSlots] counts, then p0, p1, split per node
        for (int i = threadIdx.x; i < kGridNodes * kSelectSlots; i += kThreads) s_sel[i] = 0;
        if (threadIdx.x < kGridNodes && (int)threadIdx.x < ni) {
            const cy_select_state& t = sel[(long long)j * G.nx + i0 + threadIdx.x];
            uint32_t* p = s_sel + kGridNodes * kSelectSlots + threadIdx.x;
            p[0] = t.prefix[0];
            p[kGridNodes] = t.prefix[1];
            p[2 * kGridNodes] = t.split;
        }
    }
    __syncthreads();
    int ka = -1, kb = -1;
    for (int k = 0; k < ni; ++k)
        if (s_active[k]) {
            if (ka < 0) ka = k;
            kb = k;
        }
    if (ka < 0) return;
    int a, b;
    G.rows(j, a, b);
    const int len = b - a + 1, nch = (b - a) / kUnitRows + 1;   // chunks of balanced size <= kUnitRows
    const int ya = a + (int)((long long)chunk * len / nch);
    const int nrows = a + (int)((long long)(chunk + 1) * len / nch) - ya;
    const int cs = max(G.xnode(i0 + ka) - G.h, 0), ce = min(G.xnode(i0 + kb) + G.h, G.ncols - 1);
    NAcc acc[kNodesPerWarp];
#pragma unroll
    for (int q = 0; q < kNodesPerWarp; ++q) acc[q] = {0, 0.0, 0.0};
    for (int s0 = cs; s0 <= ce; s0 += kSliceCols) {
        const int sw = min(kSliceCols, ce - s0 + 1);
        for (int r = w; r < nrows; r += kThreads / 32) {
            const uint32_t* row = img + (long long)(ya + r - row0) * row_stride + s0;
            if (kMask) {
                const uint32_t* mrow = mask + (long long)(ya + r - G.rlo) * mask_words;
                for (int c = lane; c < sw; c += 32) {
                    const int mx = s0 + c + mask_col0;
                    tile[r][c] = ((__ldg(mrow + (mx >> 5)) >> (mx & 31)) & 1u) ? __int_as_float(0x7fc00000)
                                                                              : noise_pixel(row + c, big_endian);
                }
            } else {
                for (int c = lane; c < sw; c += 32) tile[r][c] = noise_pixel(row + c, big_endian);
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kNodesPerWarp; ++q) {
            const int k = w + q * (kThreads / 32);
            if (k >= ni || !s_active[k]) continue;
            const int xk = G.xnode(i0 + k);
            const int c0 = max(xk - G.h, s0), c1 = min(xk + G.h, s0 + sw - 1);
            const double lo = s_lo[k], hi = s_hi[k], c = s_c[k];
            if constexpr (kMedian) {
                extern __shared__ uint32_t s_sel[];
                const uint32_t* p = s_sel + kGridNodes * kSelectSlots + k;
                const Select sq{p[0], p[kGridNodes], round, round > 0 ? (int)p[2 * kGridNodes] : 0, 32 - 8 * round};
                uint32_t* h = s_sel + k * kSelectSlots;
                const int nseg = (c1 - c0) / 32 + 1;   // one loop, so the warp stays converged for select_count
                for (int t = 0; t < nrows * nseg; ++t) {
                    const int r = t / nseg, x = c0 + (t - r * nseg) * 32 + lane;
                    const float f = x <= c1 ? tile[r][x - s0] : __int_as_float(0x7fc00000);
                    const double v = (double)f;
                    const bool keep = v >= lo && v <= hi;   // false for a masked pixel (NaN)
                    if (keep && round == 0) {
                        const double d = v - c;
                        acc[q].n += 1;
                        acc[q].s1 += d;
                        acc[q].s2 += d * d;
                    }
                    select_count(h, sq, keep, __float_as_uint(f));
                }
            } else {
                for (int r = 0; r < nrows; ++r)
                    for (int x = c0 + lane; x <= c1; x += 32) {
                        const double v = (double)tile[r][x - s0];
                        if (!(v >= lo && v <= hi)) continue;   // false for a masked pixel (NaN)
                        const double d = v - c;
                        acc[q].n += 1;
                        acc[q].s1 += d;
                        acc[q].s2 += d * d;
                    }
            }
        }
        __syncthreads();
    }
    if constexpr (kMedian) {   // the loop ends with a barrier: every count is in
        extern __shared__ uint32_t s_sel[];
        for (int i = threadIdx.x; i < kGridNodes * kSelectSlots; i += kThreads) {
            const int k = i / kSelectSlots;
            if (k < ni && s_active[k] && s_sel[i])
                atomicAdd(hist + ((long long)j * G.nx + i0 + k) * kSelectSlots + i % kSelectSlots, s_sel[i]);
        }
        if (round != 0) return;
    }
#pragma unroll
    for (int q = 0; q < kNodesPerWarp; ++q) {
        NAcc t = acc[q];
        for (int d = 16; d > 0; d >>= 1) {
            NAcc o;
            o.n = __shfl_down_sync(0xffffffffu, t.n, d);
            o.s1 = __shfl_down_sync(0xffffffffu, t.s1, d);
            o.s2 = __shfl_down_sync(0xffffffffu, t.s2, d);
            nacc_merge(t, o);
        }
        const int k = w + q * (kThreads / 32);
        if (lane == 0 && k < ni && s_active[k]) {
            cy_noise_partial& p = unit_out[u * kGridNodes + k];
            p.n = t.n;
            p.s1 = t.s1;
            p.s2 = t.s2;
        }
    }
}

// unit partials of each active node, folded in chunk order -> one partial per node (zero without units)
__global__ void bkg_fold_kernel(const cy_noise_partial* __restrict__ unit, const long long* __restrict__ off, Grid G,
                                const cy_noise_state* __restrict__ state, cy_noise_partial* __restrict__ out) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= (long long)G.nx * G.ny || state[n].done) return;
    const int j = (int)(n / G.nx), i = (int)(n % G.nx);
    const long long nch = (off[j + 1] - off[j]) / G.ngroups;
    NAcc a = {0, 0.0, 0.0};
    for (long long c = 0; c < nch; ++c) {
        const cy_noise_partial& p = unit[(off[j] + c * G.ngroups + i / kGridNodes) * kGridNodes + i % kGridNodes];
        const NAcc b = {p.n, p.s1, p.s2};
        nacc_merge(a, b);
    }
    out[n].n = a.n;
    out[n].s1 = a.s1;
    out[n].s2 = a.s2;
}

// bilinear weight of the finite corners, renormalised; NaN when they carry no weight
__device__ __forceinline__ float interp_corners(double v00, double v01, double v10, double v11, double w00, double w01,
                                                double w10, double w11) {
    double s = 0.0, ws = 0.0;
    if (!isnan(v00)) { s += w00 * v00; ws += w00; }
    if (!isnan(v01)) { s += w01 * v01; ws += w01; }
    if (!isnan(v10)) { s += w10 * v10; ws += w10; }
    if (!isnan(v11)) { s += w11 * v11; ws += w11; }
    return ws > 0.0 ? (float)(s / ws) : __int_as_float(0x7fc00000);
}

// the bkg and rms map values of region pixel (x, y): the corners and weights of its lattice cell, then interp_corners.
// bkg_map_kernel and snr_map_kernel both take them from here, so the two agree to the bit.
__device__ __forceinline__ void map_pixel(const cy_noise_state* __restrict__ state, const Grid& G, int x, int y,
                                          float& fb, float& fr) {
    const int i = G.nx >= 2 ? min(x / G.g, G.nx - 2) : 0, i1 = min(i + 1, G.nx - 1);   // x_i = i * g for i <= nx - 2
    const int j = G.ny >= 2 ? min((y - G.R0) / G.g, G.ny - 2) : 0, j1 = min(j + 1, G.ny - 1);
    const double t = i1 > i ? (double)(x - G.xnode(i)) / (double)(G.xnode(i1) - G.xnode(i)) : 0.0;
    const double v = j1 > j ? (double)(y - G.ynode(j)) / (double)(G.ynode(j1) - G.ynode(j)) : 0.0;
    const double w00 = (1.0 - t) * (1.0 - v), w01 = t * (1.0 - v), w10 = (1.0 - t) * v, w11 = t * v;
    const cy_noise_state &a = state[(long long)j * G.nx + i], &b = state[(long long)j * G.nx + i1];
    const cy_noise_state &c = state[(long long)j1 * G.nx + i], &d = state[(long long)j1 * G.nx + i1];
    fb = interp_corners(a.bkg, b.bkg, c.bkg, d.bkg, w00, w01, w10, w11);
    fr = interp_corners(a.rms, b.rms, c.rms, d.rms, w00, w01, w10, w11);
}

// one thread per map pixel: blockIdx.x = row - row_begin, blockIdx.y * blockDim.x + threadIdx.x = column
__global__ void bkg_map_kernel(const cy_noise_state* __restrict__ state, Grid G, int row_begin,
                               uint32_t* __restrict__ bkg, uint32_t* __restrict__ rms) {
    const int x = blockIdx.y * blockDim.x + threadIdx.x;
    if (x >= G.ncols) return;
    float fb, fr;
    map_pixel(state, G, x, row_begin + blockIdx.x, fb, fr);
    const long long o = (long long)blockIdx.x * G.ncols + x;
    bkg[o] = __byte_perm(__float_as_uint(fb), 0, 0x0123);   // FITS byte order
    rms[o] = __byte_perm(__float_as_uint(fr), 0, 0x0123);
}

// background-subtracted and S/N maps (cy_bkg_grid_snr_maps), the grid of bkg_map_kernel: each thread reads its image
// pixel once (a warp reads 32 adjacent words of one row) and writes res = v - bkg and snr = (v - bkg) / rms, both in
// fp64 and rounded once.  NaN: a masked pixel or a NaN bkg in both maps; a NaN or non-positive rms in snr only.
__global__ void snr_map_kernel(const uint32_t* __restrict__ img, long long row_stride, int big_endian, int row0,
                               const cy_noise_state* __restrict__ state, Grid G, int row_begin,
                               uint32_t* __restrict__ res, uint32_t* __restrict__ snr) {
    const int x = blockIdx.y * blockDim.x + threadIdx.x;
    if (x >= G.ncols) return;
    const int y = row_begin + blockIdx.x;
    const float v = noise_pixel(img + (long long)(y - row0) * row_stride + x, big_endian);
    float fb, fr;
    map_pixel(state, G, x, y, fb, fr);
    float r = __int_as_float(0x7fc00000), s = r;
    if (!isnan(v) && !isnan(fb)) {
        const double d = (double)v - (double)fb;
        r = (float)d;
        if (fr > 0.0f) s = (float)(d / (double)fr);   // false for NaN
    }
    const long long o = (long long)blockIdx.x * G.ncols + x;
    res[o] = __byte_perm(__float_as_uint(r), 0, 0x0123);   // FITS byte order
    snr[o] = __byte_perm(__float_as_uint(s), 0, 0x0123);
}

// ---------------------------------------------------------------------------------------------- source mask
// The union M of the catalog boxes as a bit mask (cy_source_mask): the units of measure_units_scan_kernel with grow = 0,
// one CTA per unit; each thread ORs the bits of one (row, word) of the unit's rows into the mask.  OR does not depend on
// the order, so overlapping boxes give the same bits whatever CTA runs first.
__global__ void __launch_bounds__(kThreads) source_mask_kernel(const cy_source* __restrict__ src, int nsrc, int ncols,
                                                               int row_begin, int row_end,
                                                               const long long* __restrict__ off,
                                                               uint32_t* __restrict__ mask) {
    const long long u = blockIdx.x;
    const int s = unit_source(off, nsrc, u);
    Box b;
    source_box(src[s], 0, ncols, row_begin, row_end, b);
    const int ya = b.y0 + (int)(u - off[s]) * kUnitRows;
    const int nrows = min(b.y1, ya + kUnitRows - 1) - ya + 1;
    const int w0 = b.x0 >> 5, nw = (b.x1 >> 5) - w0 + 1, words = (ncols + 31) >> 5;
    for (int t = threadIdx.x; t < nrows * nw; t += kThreads) {
        const int r = t / nw, w = w0 + t % nw;
        const int lo = max(b.x0 - 32 * w, 0), hi = min(b.x1 - 32 * w, 31);   // bits lo..hi of word w
        const uint32_t bits = (hi - lo == 31 ? 0xffffffffu : ((1u << (hi - lo + 1)) - 1u)) << lo;
        atomicOr(mask + (long long)(ya + r - row_begin) * words + w, bits);
    }
}

// ---------------------------------------------------------------------------------------------- hole fill
// Node classes of the fill (cy_bkg_grid_fill): a value (finite after clipping, or filled), an unfilled hole, blank.
enum { kFillValue = 0, kFillHole = 1, kFillBlank = 2 };
struct FillNode {
    double bkg, rms;
    int cls;
};

// probe state: pass 0 for the nodes without a value (nbkg = 0), done for the others; *nprobe counts the former
__global__ void bkg_probe_init_kernel(const cy_noise_state* __restrict__ state, int nodes,
                                      cy_noise_state* __restrict__ probe, int* __restrict__ nprobe) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nodes) return;
    cy_noise_state t;
    t.lo = -INFINITY;
    t.hi = INFINITY;
    t.c = 0.0;
    t.bkg = t.rms = __longlong_as_double(0x7ff8000000000000ll);
    t.nbkg = 0;
    t.iters = 0;
    t.done = state[n].nbkg > 0;
    if (!t.done) atomicAdd(nprobe, 1);
    probe[n] = t;
}

// final node states + the probe partials [world][nodes] (read for the nodes with nbkg = 0 only) -> fill nodes
__global__ void bkg_fill_classify_kernel(const cy_noise_partial* __restrict__ part, int world, int nodes,
                                         const cy_noise_state* __restrict__ state, FillNode* __restrict__ out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nodes) return;
    FillNode f;
    f.bkg = state[n].bkg;
    f.rms = state[n].rms;
    f.cls = kFillValue;
    if (state[n].nbkg == 0) {
        long long k = 0;
        for (int r = 0; r < world; ++r) k += part[(long long)r * nodes + n].n;
        f.cls = k > 0 ? kFillHole : kFillBlank;
    }
    out[n] = f;
}

// one ring: every hole with a valued node among its 8 neighbours in `a` takes the mean of their values (summed in
// row-major neighbour order) -> b; *changed counts the nodes filled in this ring
__global__ void bkg_fill_ring_kernel(const FillNode* __restrict__ a, int nx, int ny, FillNode* __restrict__ b,
                                     int* __restrict__ changed) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= (long long)nx * ny) return;
    FillNode f = a[n];
    if (f.cls == kFillHole) {
        const int j = (int)(n / nx), i = (int)(n % nx);
        double sb = 0.0, sr = 0.0;
        int k = 0;
        for (int dj = -1; dj <= 1; ++dj)
            for (int di = -1; di <= 1; ++di) {
                const int jj = j + dj, ii = i + di;
                if ((dj == 0 && di == 0) || jj < 0 || jj >= ny || ii < 0 || ii >= nx) continue;
                const FillNode& q = a[(long long)jj * nx + ii];
                if (q.cls != kFillValue) continue;
                sb += q.bkg;
                sr += q.rms;
                ++k;
            }
        if (k > 0) {
            f.bkg = sb / k;
            f.rms = sr / k;
            f.cls = kFillValue;
            atomicAdd(changed, 1);
        }
    }
    b[n] = f;
}

// filled values -> the node states (nbkg stays 0, so a filled node can be recognised)
__global__ void bkg_fill_store_kernel(const FillNode* __restrict__ a, int nodes, cy_noise_state* __restrict__ state) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nodes || state[n].nbkg > 0 || a[n].cls != kFillValue) return;
    state[n].bkg = a[n].bkg;
    state[n].rms = a[n].rms;
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
    measure_units_scan_kernel<<<1, kScanThreads, 0, st>>>(src, nsrc, 0, ncols, row_begin, row_end, off);
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

extern "C" int cy_noise_init(const cy_source* src, int nsrc, int ncols, int row_begin, int row_end, int frame,
                             cy_noise_state* state, long long* unit_off, long long* units, uintptr_t stream) {
    if (nsrc < 0 || ncols <= 0 || row_end < row_begin || frame < 1 || !units)
        return set_error(CY_ERR_INVALID, "cy_noise_init: invalid image geometry, row range or frame width");
    *units = 0;
    if (nsrc == 0) return CY_OK;
    if (!src || !state || !unit_off) return set_error(CY_ERR_INVALID, "cy_noise_init: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    noise_init_kernel<<<(nsrc + 255) / 256, 256, 0, st>>>(nsrc, state);
    measure_units_scan_kernel<<<1, kScanThreads, 0, st>>>(src, nsrc, frame, ncols, row_begin, row_end, unit_off);
    long long n = 0;   // the unit count is data dependent: bring it to the host
    cudaMemcpyAsync(&n, unit_off + nsrc, sizeof(long long), cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_noise_init: %s", cudaGetErrorString(e));
    if (n > 2147483647ll) return set_error(CY_ERR_INVALID, "cy_noise_init: %lld work units exceed one grid", n);
    *units = n;
    return CY_OK;
}

// sel == nullptr: a pass of the mean; otherwise round `round` of a median pass (hist zeroed, then counted; the moment
// partials are written in round 0 only)
static int noise_pass(const char* fn, const void* img, long long row_stride, int big_endian, int row0, int ncols,
                      const cy_source* src, int nsrc, int row_begin, int row_end, int frame, const long long* unit_off,
                      long long units, const cy_noise_state* state, cy_noise_partial* partials, const uint32_t* mask,
                      uintptr_t stream, const cy_select_state* sel = nullptr, int round = 0, uint32_t* hist = nullptr) {
    if (nsrc < 0 || ncols <= 0 || row_stride < ncols || row_begin < row0 || row_end < row_begin || frame < 1 ||
        units < 0 || units > 2147483647ll || round < 0 || round >= kSelectRounds)
        return set_error(CY_ERR_INVALID, "%s: invalid image geometry, row range, frame, unit count or round", fn);
    if (nsrc == 0) return CY_OK;
    if (!src || !unit_off || !state || !partials || (units > 0 && !img))
        return set_error(CY_ERR_INVALID, "%s: null argument", fn);
    cudaStream_t st = (cudaStream_t)stream;
    if (sel) CY_CUDA_CHECK(cudaMemsetAsync(hist, 0, (size_t)nsrc * kSelectSlots * sizeof(uint32_t), st));
    const bool moments = !sel || round == 0;
    cy_noise_partial* unit = nullptr;
    if (moments && units > 0 && cudaMallocAsync(&unit, (size_t)units * sizeof(cy_noise_partial), st) != cudaSuccess)
        return set_error(CY_ERR_NOMEM, "%s: no memory for %lld unit partials", fn, units);
    const uint32_t* I = (const uint32_t*)img;
    if (units > 0 && sel && mask)
        noise_unit_kernel<true, true><<<(unsigned)units, kThreads, 0, st>>>(I, row_stride, big_endian, row0, ncols,
                                                                            src, nsrc, row_begin, row_end, frame,
                                                                            unit_off, state, unit, mask, sel, round,
                                                                            hist);
    else if (units > 0 && sel)
        noise_unit_kernel<false, true><<<(unsigned)units, kThreads, 0, st>>>(I, row_stride, big_endian, row0, ncols,
                                                                             src, nsrc, row_begin, row_end, frame,
                                                                             unit_off, state, unit, nullptr, sel,
                                                                             round, hist);
    else if (units > 0 && mask)
        noise_unit_kernel<true><<<(unsigned)units, kThreads, 0, st>>>((const uint32_t*)img, row_stride, big_endian,
                                                                      row0, ncols, src, nsrc, row_begin, row_end,
                                                                      frame, unit_off, state, unit, mask);
    else if (units > 0)
        noise_unit_kernel<false><<<(unsigned)units, kThreads, 0, st>>>((const uint32_t*)img, row_stride, big_endian,
                                                                       row0, ncols, src, nsrc, row_begin, row_end,
                                                                       frame, unit_off, state, unit, nullptr);
    if (moments) noise_fold_kernel<<<(nsrc + 255) / 256, 256, 0, st>>>(unit, unit_off, nsrc, state, partials);
    const cudaError_t e = cudaGetLastError();
    if (unit) cudaFreeAsync(unit, st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "%s: %s", fn, cudaGetErrorString(e));
    return CY_OK;
}

extern "C" int cy_noise_pass(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                             const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                             const long long* unit_off, long long units, const cy_noise_state* state,
                             cy_noise_partial* partials, uintptr_t stream) {
    return noise_pass("cy_noise_pass", img, row_stride, big_endian, row0, ncols, src, nsrc, row_begin, row_end, frame,
                      unit_off, units, state, partials, nullptr, stream);
}

extern "C" int cy_noise_pass_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                    const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                                    const long long* unit_off, long long units, const cy_noise_state* state,
                                    cy_noise_partial* partials, const uint32_t* mask, uintptr_t stream) {
    if (units > 0 && row_end > row_begin && !mask)
        return set_error(CY_ERR_INVALID, "cy_noise_pass_masked: null mask");
    return noise_pass("cy_noise_pass_masked", img, row_stride, big_endian, row0, ncols, src, nsrc, row_begin, row_end,
                      frame, unit_off, units, state, partials, row_end > row_begin ? mask : nullptr, stream);
}

static int median_args(const char* fn, const cy_select_state* sel, uint32_t* hist) {
    if (!sel || !hist) return set_error(CY_ERR_INVALID, "%s: null select state or histogram", fn);
    return CY_OK;
}

extern "C" int cy_noise_pass_median(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                    const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                                    const long long* unit_off, long long units, const cy_noise_state* state,
                                    const cy_select_state* sel, int round, cy_noise_partial* partials,
                                    uint32_t* hist, uintptr_t stream) {
    if (nsrc > 0 && median_args("cy_noise_pass_median", sel, hist)) return CY_ERR_INVALID;
    return noise_pass("cy_noise_pass_median", img, row_stride, big_endian, row0, ncols, src, nsrc, row_begin, row_end,
                      frame, unit_off, units, state, partials, nullptr, stream, sel, round, hist);
}

extern "C" int cy_noise_pass_median_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                           const cy_source* src, int nsrc, int row_begin, int row_end, int frame,
                                           const long long* unit_off, long long units, const cy_noise_state* state,
                                           const cy_select_state* sel, int round, cy_noise_partial* partials,
                                           uint32_t* hist, const uint32_t* mask, uintptr_t stream) {
    if (units > 0 && row_end > row_begin && !mask)
        return set_error(CY_ERR_INVALID, "cy_noise_pass_median_masked: null mask");
    if (nsrc > 0 && median_args("cy_noise_pass_median_masked", sel, hist)) return CY_ERR_INVALID;
    return noise_pass("cy_noise_pass_median_masked", img, row_stride, big_endian, row0, ncols, src, nsrc, row_begin,
                      row_end, frame, unit_off, units, state, partials, row_end > row_begin ? mask : nullptr, stream,
                      sel, round, hist);
}

extern "C" int cy_median_update(const cy_noise_partial* partials, int world, const uint32_t* hist, int n,
                                cy_noise_state* state, cy_select_state* sel, int round, int* active,
                                uintptr_t stream) {
    if (world < 1 || n < 0 || round < 0 || round >= kSelectRounds || (round == kSelectRounds - 1 && !active))
        return set_error(CY_ERR_INVALID, "cy_median_update: invalid arguments");
    if (active) *active = 0;
    if (n == 0) return CY_OK;
    if (!partials || !hist || !state || !sel) return set_error(CY_ERR_INVALID, "cy_median_update: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (round < kSelectRounds - 1) {
        median_update_kernel<<<(n + 255) / 256, 256, 0, st>>>(partials, world, hist, n, state, sel, round, nullptr);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_median_update: %s", cudaGetErrorString(e));
        return CY_OK;
    }
    int* cnt = nullptr;
    CY_CUDA_CHECK(cudaMallocAsync(&cnt, 2 * sizeof(int), st));
    cudaMemsetAsync(cnt, 0, 2 * sizeof(int), st);
    median_update_kernel<<<(n + 255) / 256, 256, 0, st>>>(partials, world, hist, n, state, sel, round, cnt);
    int h[2] = {0, 0};
    cudaMemcpyAsync(h, cnt, 2 * sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(cnt, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_median_update: %s", cudaGetErrorString(e));
    if (h[1] > 0)
        return set_error(CY_ERR_INVALID, "cy_median_update: %d frames or node boxes keep 2^32 pixels or more", h[1]);
    *active = h[0];
    return CY_OK;
}

extern "C" int cy_noise_update(const cy_noise_partial* partials, int world, int nsrc, cy_noise_state* state,
                               int* active, uintptr_t stream) {
    if (world < 1 || nsrc < 0 || !active) return set_error(CY_ERR_INVALID, "cy_noise_update: invalid arguments");
    *active = 0;
    if (nsrc == 0) return CY_OK;
    if (!partials || !state) return set_error(CY_ERR_INVALID, "cy_noise_update: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int* cnt = nullptr;
    CY_CUDA_CHECK(cudaMallocAsync(&cnt, sizeof(int), st));
    cudaMemsetAsync(cnt, 0, sizeof(int), st);
    noise_update_kernel<<<(nsrc + 255) / 256, 256, 0, st>>>(partials, world, nsrc, state, cnt);
    int n = 0;
    cudaMemcpyAsync(&n, cnt, sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(cnt, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_noise_update: %s", cudaGetErrorString(e));
    *active = n;
    return CY_OK;
}

extern "C" int cy_bkg_grid_init(int ncols, int R0, int R1, int row_begin, int row_end, int box, int grid,
                                cy_noise_state* state, long long* unit_off, long long* units, uintptr_t stream) {
    Grid G;
    if (!units || !make_grid(ncols, R0, R1, row_begin, row_end, box, grid, G))
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_init: invalid region, row range, box (odd, >= 3) or grid (>= 1)");
    *units = 0;
    if (!state || !unit_off) return set_error(CY_ERR_INVALID, "cy_bkg_grid_init: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const long long nodes = (long long)G.nx * G.ny;
    noise_init_kernel<<<(unsigned)((nodes + 255) / 256), 256, 0, st>>>((int)nodes, state);
    bkg_units_scan_kernel<<<1, kScanThreads, 0, st>>>(G, unit_off);
    long long n = 0;   // the unit count is data dependent: bring it to the host
    cudaMemcpyAsync(&n, unit_off + G.ny, sizeof(long long), cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_bkg_grid_init: %s", cudaGetErrorString(e));
    if (n > 2147483647ll) return set_error(CY_ERR_INVALID, "cy_bkg_grid_init: %lld work units exceed one grid", n);
    *units = n;
    return CY_OK;
}

// sel == nullptr: a pass of the mean; otherwise round `round` of a median pass, as for noise_pass
static int bkg_grid_pass(const char* fn, const void* img, long long row_stride, int big_endian, int row0, int ncols,
                         int R0, int R1, int row_begin, int row_end, int box, int grid, const long long* unit_off,
                         long long units, const cy_noise_state* state, cy_noise_partial* partials,
                         const uint32_t* mask, int mask_ncols, int mask_col0, uintptr_t stream,
                         const cy_select_state* sel = nullptr, int round = 0, uint32_t* hist = nullptr) {
    Grid G;
    if (!make_grid(ncols, R0, R1, row_begin, row_end, box, grid, G) || row_stride < ncols || row_begin < row0 ||
        units < 0 || units > 2147483647ll || round < 0 || round >= kSelectRounds)
        return set_error(CY_ERR_INVALID, "%s: invalid image geometry, region, box, grid, unit count or round", fn);
    if (!unit_off || !state || !partials || (units > 0 && !img))
        return set_error(CY_ERR_INVALID, "%s: null argument", fn);
    cudaStream_t st = (cudaStream_t)stream;
    const long long nodes = (long long)G.nx * G.ny;
    if (sel) CY_CUDA_CHECK(cudaMemsetAsync(hist, 0, (size_t)nodes * kSelectSlots * sizeof(uint32_t), st));
    const bool moments = !sel || round == 0;
    cy_noise_partial* unit = nullptr;
    if (moments && units > 0 &&
        cudaMallocAsync(&unit, (size_t)units * kGridNodes * sizeof(cy_noise_partial), st) != cudaSuccess)
        return set_error(CY_ERR_NOMEM, "%s: no memory for %lld unit partials", fn, units * kGridNodes);
    const uint32_t* I = (const uint32_t*)img;
    const int words = (mask_ncols + 31) >> 5;
    if (units > 0 && sel) {
        auto k = mask ? bkg_unit_kernel<true, true> : bkg_unit_kernel<false, true>;
        CY_CUDA_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kBkgSelectSmem));
        k<<<(unsigned)units, kThreads, kBkgSelectSmem, st>>>(I, row_stride, big_endian, row0, G, unit_off, state, unit,
                                                            mask, mask ? words : 0, mask ? mask_col0 : 0, sel, round,
                                                            hist);
    } else if (units > 0 && mask)
        bkg_unit_kernel<true><<<(unsigned)units, kThreads, 0, st>>>((const uint32_t*)img, row_stride, big_endian, row0,
                                                                    G, unit_off, state, unit, mask,
                                                                    (mask_ncols + 31) >> 5, mask_col0);
    else if (units > 0)
        bkg_unit_kernel<false><<<(unsigned)units, kThreads, 0, st>>>((const uint32_t*)img, row_stride, big_endian, row0,
                                                                     G, unit_off, state, unit, nullptr, 0, 0);
    if (moments) bkg_fold_kernel<<<(unsigned)((nodes + 255) / 256), 256, 0, st>>>(unit, unit_off, G, state, partials);
    const cudaError_t e = cudaGetLastError();
    if (unit) cudaFreeAsync(unit, st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "%s: %s", fn, cudaGetErrorString(e));
    return CY_OK;
}

extern "C" int cy_bkg_grid_pass(const void* img, long long row_stride, int big_endian, int row0, int ncols, int R0,
                                int R1, int row_begin, int row_end, int box, int grid, const long long* unit_off,
                                long long units, const cy_noise_state* state, cy_noise_partial* partials,
                                uintptr_t stream) {
    return bkg_grid_pass("cy_bkg_grid_pass", img, row_stride, big_endian, row0, ncols, R0, R1, row_begin, row_end, box,
                         grid, unit_off, units, state, partials, nullptr, 0, 0, stream);
}

extern "C" int cy_bkg_grid_pass_masked(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                       int R0, int R1, int row_begin, int row_end, int box, int grid,
                                       const long long* unit_off, long long units, const cy_noise_state* state,
                                       cy_noise_partial* partials, const uint32_t* mask, int mask_ncols,
                                       int mask_col0, uintptr_t stream) {
    if (mask_col0 < 0 || ncols <= 0 || mask_ncols < 1 || (long long)mask_col0 + ncols > mask_ncols)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_pass_masked: the region's columns [%d, %lld) are not inside the "
                         "mask's %d columns", mask_col0, (long long)mask_col0 + ncols, mask_ncols);
    if (units > 0 && row_end > row_begin && !mask)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_pass_masked: null mask");
    return bkg_grid_pass("cy_bkg_grid_pass_masked", img, row_stride, big_endian, row0, ncols, R0, R1, row_begin,
                         row_end, box, grid, unit_off, units, state, partials, row_end > row_begin ? mask : nullptr,
                         mask_ncols, mask_col0, stream);
}

extern "C" int cy_bkg_grid_pass_median(const void* img, long long row_stride, int big_endian, int row0, int ncols,
                                       int R0, int R1, int row_begin, int row_end, int box, int grid,
                                       const long long* unit_off, long long units, const cy_noise_state* state,
                                       const cy_select_state* sel, int round, cy_noise_partial* partials,
                                       uint32_t* hist, uintptr_t stream) {
    if (median_args("cy_bkg_grid_pass_median", sel, hist)) return CY_ERR_INVALID;
    return bkg_grid_pass("cy_bkg_grid_pass_median", img, row_stride, big_endian, row0, ncols, R0, R1, row_begin,
                         row_end, box, grid, unit_off, units, state, partials, nullptr, 0, 0, stream, sel, round,
                         hist);
}

extern "C" int cy_bkg_grid_pass_median_masked(const void* img, long long row_stride, int big_endian, int row0,
                                              int ncols, int R0, int R1, int row_begin, int row_end, int box, int grid,
                                              const long long* unit_off, long long units,
                                              const cy_noise_state* state, const cy_select_state* sel, int round,
                                              cy_noise_partial* partials, uint32_t* hist, const uint32_t* mask,
                                              int mask_ncols, int mask_col0, uintptr_t stream) {
    if (mask_col0 < 0 || ncols <= 0 || mask_ncols < 1 || (long long)mask_col0 + ncols > mask_ncols)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_pass_median_masked: the region's columns [%d, %lld) are not "
                         "inside the mask's %d columns", mask_col0, (long long)mask_col0 + ncols, mask_ncols);
    if (units > 0 && row_end > row_begin && !mask)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_pass_median_masked: null mask");
    if (median_args("cy_bkg_grid_pass_median_masked", sel, hist)) return CY_ERR_INVALID;
    return bkg_grid_pass("cy_bkg_grid_pass_median_masked", img, row_stride, big_endian, row0, ncols, R0, R1,
                         row_begin, row_end, box, grid, unit_off, units, state, partials,
                         row_end > row_begin ? mask : nullptr, mask_ncols, mask_col0, stream, sel, round, hist);
}

extern "C" int cy_bkg_grid_maps(const cy_noise_state* state, int ncols, int R0, int R1, int row_begin, int row_end,
                                int box, int grid, void* bkg, void* rms, uintptr_t stream) {
    Grid G;
    if (!make_grid(ncols, R0, R1, row_begin, row_end, box, grid, G) || (ncols + 255) / 256 > 65535)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_maps: invalid region, row range, box or grid");
    if (row_end == row_begin) return CY_OK;
    if (!state || !bkg || !rms) return set_error(CY_ERR_INVALID, "cy_bkg_grid_maps: null argument");
    bkg_map_kernel<<<dim3((unsigned)(row_end - row_begin), (unsigned)((ncols + 255) / 256)), 256, 0,
                     (cudaStream_t)stream>>>(state, G, row_begin, (uint32_t*)bkg, (uint32_t*)rms);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_bkg_grid_maps: %s", cudaGetErrorString(e));
    return CY_OK;
}

extern "C" int cy_bkg_grid_snr_maps(const cy_noise_state* state, const void* img, long long row_stride, int big_endian,
                                    int row0, int ncols, int R0, int R1, int row_begin, int row_end, int box, int grid,
                                    void* res, void* snr, uintptr_t stream) {
    Grid G;
    if (!make_grid(ncols, R0, R1, row_begin, row_end, box, grid, G) || (ncols + 255) / 256 > 65535 ||
        row_stride < ncols || row_begin < row0)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_snr_maps: invalid image geometry, region, row range, box or grid");
    if (row_end == row_begin) return CY_OK;
    if (!state || !img || !res || !snr) return set_error(CY_ERR_INVALID, "cy_bkg_grid_snr_maps: null argument");
    snr_map_kernel<<<dim3((unsigned)(row_end - row_begin), (unsigned)((ncols + 255) / 256)), 256, 0,
                     (cudaStream_t)stream>>>((const uint32_t*)img, row_stride, big_endian, row0, state, G, row_begin,
                                             (uint32_t*)res, (uint32_t*)snr);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_bkg_grid_snr_maps: %s", cudaGetErrorString(e));
    return CY_OK;
}

extern "C" int cy_source_mask(const cy_source* src, int nsrc, int ncols, int row_begin, int row_end, uint32_t* mask,
                              uintptr_t stream) {
    if (nsrc < 0 || ncols <= 0 || row_end < row_begin)
        return set_error(CY_ERR_INVALID, "cy_source_mask: invalid source count, column count or row range");
    const long long words = (long long)(row_end - row_begin) * ((ncols + 31) >> 5);
    if (words == 0) return CY_OK;
    if (!mask || (nsrc > 0 && !src)) return set_error(CY_ERR_INVALID, "cy_source_mask: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    CY_CUDA_CHECK(cudaMemsetAsync(mask, 0, (size_t)words * sizeof(uint32_t), st));
    if (nsrc == 0) return CY_OK;
    long long* off = nullptr;
    CY_CUDA_CHECK(cudaMallocAsync(&off, (size_t)(nsrc + 1) * sizeof(long long), st));
    measure_units_scan_kernel<<<1, kScanThreads, 0, st>>>(src, nsrc, 0, ncols, row_begin, row_end, off);
    long long units = 0;   // the unit count is data dependent: bring it to the host
    cudaMemcpyAsync(&units, off + nsrc, sizeof(long long), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess && units > 2147483647ll) {
        cudaFreeAsync(off, st);
        return set_error(CY_ERR_INVALID, "cy_source_mask: %lld work units exceed one grid", units);
    }
    if (e == cudaSuccess && units > 0)
        source_mask_kernel<<<(unsigned)units, kThreads, 0, st>>>(src, nsrc, ncols, row_begin, row_end, off, mask);
    if (e == cudaSuccess) e = cudaGetLastError();
    cudaFreeAsync(off, st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_source_mask: %s", cudaGetErrorString(e));
    return CY_OK;
}

extern "C" int cy_bkg_grid_probe_init(const cy_noise_state* state, int nodes, cy_noise_state* probe, int* nprobe,
                                      uintptr_t stream) {
    if (nodes < 1 || !nprobe) return set_error(CY_ERR_INVALID, "cy_bkg_grid_probe_init: invalid arguments");
    *nprobe = 0;
    if (!state || !probe) return set_error(CY_ERR_INVALID, "cy_bkg_grid_probe_init: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int* cnt = nullptr;
    CY_CUDA_CHECK(cudaMallocAsync(&cnt, sizeof(int), st));
    cudaMemsetAsync(cnt, 0, sizeof(int), st);
    bkg_probe_init_kernel<<<(nodes + 255) / 256, 256, 0, st>>>(state, nodes, probe, cnt);
    int n = 0;
    cudaMemcpyAsync(&n, cnt, sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(cnt, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_bkg_grid_probe_init: %s", cudaGetErrorString(e));
    *nprobe = n;
    return CY_OK;
}

extern "C" int cy_bkg_grid_fill(const cy_noise_partial* probe_partials, int world, int nx, int ny,
                                cy_noise_state* state, int* filled, uintptr_t stream) {
    if (world < 1 || nx < 1 || ny < 1 || (long long)nx * ny > 2147483647ll || !filled)
        return set_error(CY_ERR_INVALID, "cy_bkg_grid_fill: invalid arguments");
    *filled = 0;
    if (!probe_partials || !state) return set_error(CY_ERR_INVALID, "cy_bkg_grid_fill: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int nodes = nx * ny, blocks = (nodes + 255) / 256;
    FillNode* buf = nullptr;
    int* cnt = nullptr;
    CY_CUDA_CHECK(cudaMallocAsync(&buf, 2 * (size_t)nodes * sizeof(FillNode), st));
    if (cudaMallocAsync(&cnt, sizeof(int), st) != cudaSuccess) {
        cudaFreeAsync(buf, st);
        return set_error(CY_ERR_NOMEM, "cy_bkg_grid_fill: no memory for the ring counter");
    }
    FillNode *a = buf, *b = buf + nodes;
    bkg_fill_classify_kernel<<<blocks, 256, 0, st>>>(probe_partials, world, nodes, state, a);
    cudaError_t e = cudaSuccess;
    int total = 0;
    for (;;) {   // a ring fills at least one node or ends the fill: at most nodes + 1 rings
        cudaMemsetAsync(cnt, 0, sizeof(int), st);
        bkg_fill_ring_kernel<<<blocks, 256, 0, st>>>(a, nx, ny, b, cnt);
        int changed = 0;
        cudaMemcpyAsync(&changed, cnt, sizeof(int), cudaMemcpyDeviceToHost, st);
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess || changed == 0) break;
        total += changed;
        FillNode* t = a;
        a = b;
        b = t;
    }
    if (e == cudaSuccess) {
        bkg_fill_store_kernel<<<blocks, 256, 0, st>>>(a, nodes, state);
        e = cudaGetLastError();
    }
    cudaFreeAsync(cnt, st);
    cudaFreeAsync(buf, st);
    if (e != cudaSuccess) return set_error(CY_ERR_CUDA, "cy_bkg_grid_fill: %s", cudaGetErrorString(e));
    *filled = total;
    return CY_OK;
}
