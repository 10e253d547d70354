// warp.cu — general grid warp (SURVEY section 8f row 4): the band-interleaved WGS-84 ortho cube resampled onto the
// Sentinel-2 UTM 60 m grid with GDAL's cubic kernel — the job nc_to_envi hands to a `gdalwarp -r cubic -srcnodata
// -9999 -dstnodata -9999 -t_srs <S2 CRS> -te ... -ts ...` subprocess (EMIT_data/emit_proj.py:876-940) — and the
// same-CRS affine case of the notebook's reproject_stack_to_grid.  Parity with GDAL / PROJ is UNPINNED (neither is
// installable in the build image); the algorithm restated is documented in oracle/warp.py:
//   * destination pixel centre -> projected coordinates (destination geotransform) -> lon / lat by the inverse
//     transverse Mercator (Krueger series to n^6, Karney 2011; fp64, one destination pixel per lane) -> source pixel
//     coordinates (inverse source geotransform); exact per pixel (gdalwarp -et 0);
//   * separable cubic-convolution (a = -0.5) or bilinear weights, radius widened to ceil(r / scale) with the argument
//     scaled where the destination is coarser than the source; taps outside the source or equal to nodata are
//     skipped PER BAND and the sum is divided by the accumulated weight; centre outside the source or accumulated
//     weight < 1e-6 -> dst_nodata.  NaN is an ordinary value.
// Kernels 1 and 2 (bilinear, cubic) take the source coordinates of every destination pixel from the caller's workspace
// (warp_coords_kernel) and then run one of three kernels: warp_quad_kernel (TMA-staged 2 x 2 pixel blocks, the default)
// or warp_lane_kernel (records that are not 16-byte aligned) for filter radii up to 4; warp_exact_kernel (fp64 straight
// from global memory) for wider filters and for sources of 2^32 pixels or more.  The two fast kernels classify what they
// stage (no nodata -> plain FMAs under a uniform weight sum; all nodata -> skipped; band-specific nodata -> exact
// per-element weights) and list the pixels whose fp32 quotient is ill-conditioned; warp_exact_kernel recomputes those.
#include <cuda.h>
#include <math.h>
#include <stdlib.h>

#include "hsr_common.cuh"

namespace hsr {

namespace {

constexpr int WARPS = 8;        // warps per CTA
constexpr int MAX_TAPS = 16;    // taps per axis: radius <= 8, i.e. scale >= 0.25 for cubic

struct WarpParams {
    const float* src;
    long long Hs, Ws, src_pix_stride;
    int bands;
    double dgt[6];              // destination geotransform
    double sx0, sy0, inv[4];    // source: px = inv0 * (X - sx0) + inv1 * (Y - sy0); py = inv2 * (X - sx0) + inv3 * (Y - sy0)
    int utm;                    // 1: destination is transverse Mercator (UTM), source is lon / lat in degrees
    double lon0_deg, false_northing, k0A_inv, e, e2m, beta[6];
    long long Hd, Wd;
    float* dst;
    long long dst_pix_stride;
    int has_nodata;
    float nodata, dst_nodata;
    int kind;                   // 0 nearest, 1 bilinear, 2 cubic, 3 average
    int rx, ry;                 // radius in taps per axis
    double fx, fy;              // min(scale, 1) per axis
    double* coords;             // source coordinates of every destination pixel (warp_coords_kernel)
    unsigned long long* redo_list;   // quad / lane kernel -> warp_exact_kernel: (pixel << 8 | band group) of ill-conditioned quotients
    unsigned int* redo_count;
    unsigned int redo_cap;
};

__host__ __device__ __forceinline__ double taup_of(double tau, double e) {
    const double s1 = sqrt(1.0 + tau * tau);
    const double sigma = sinh(e * atanh(e * tau / s1));
    return tau * sqrt(1.0 + sigma * sigma) - sigma * s1;
}

// centre of destination pixel (col, row) -> source pixel coordinates (pixel (i, j) has its centre at (i + .5, j + .5))
__host__ __device__ inline void dst_to_src(const WarpParams& P, double c, double r, double& px, double& py) {
    double X = P.dgt[0] + c * P.dgt[1] + r * P.dgt[2];
    double Y = P.dgt[3] + c * P.dgt[4] + r * P.dgt[5];
    if (P.utm) {
        const double xi = (Y - P.false_northing) * P.k0A_inv, eta = (X - 500000.0) * P.k0A_inv;
        double xip = xi, etap = eta;
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            double s, co;
            sincos(2.0 * (j + 1) * xi, &s, &co);
            const double a = 2.0 * (j + 1) * eta;
            xip -= P.beta[j] * s * cosh(a);
            etap -= P.beta[j] * co * sinh(a);
        }
        const double sh = sinh(etap), cx = cos(xip);
        const double tp = sin(xip) / sqrt(sh * sh + cx * cx);
        const double lam = atan2(sh, cx);
        double tau = tp;
        for (int it = 0; it < 4; ++it) {     // Newton on tau'(tau) = tp; quadratic, 2-3 steps reach 1 ulp
            const double ti = taup_of(tau, P.e);
            tau += (tp - ti) / sqrt(1.0 + ti * ti) * (1.0 + P.e2m * tau * tau) / (P.e2m * sqrt(1.0 + tau * tau));
        }
        X = lam * (180.0 / 3.14159265358979323846) + P.lon0_deg;
        Y = atan(tau) * (180.0 / 3.14159265358979323846);
    }
    const double dx = X - P.sx0, dy = Y - P.sy0;
    px = P.inv[0] * dx + P.inv[1] * dy;
    py = P.inv[2] * dx + P.inv[3] * dy;
}

__device__ __forceinline__ double tap_weight(int kind, double x) {
    const double ax = fabs(x);
    double w;
    if (kind == 2) {    // GWKCubic, a = -0.5
        if (ax <= 1.0) w = (1.5 * ax - 2.5) * ax * ax + 1.0;
        else if (ax <= 2.0) w = ((-0.5 * ax + 2.5) * ax - 4.0) * ax + 2.0;
        else w = 0.0;
    } else {
        w = ax <= 1.0 ? 1.0 - ax : 0.0;
    }
    return w;
}

__global__ void __launch_bounds__(32 * WARPS) warp_coords_kernel(const WarpParams P) {
    const long long n = P.Hd * P.Wd;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < n; o += (long long)gridDim.x * blockDim.x) {
        const long long r = o / P.Wd, c = o - r * P.Wd;
        double px, py;
        dst_to_src(P, (double)c + 0.5, (double)r + 0.5, px, py);
        P.coords[2 * o] = px;
        P.coords[2 * o + 1] = py;
    }
}

// Point kernels: kind 0 = nearest neighbour (GWKNearest: the source pixel holding the destination centre), kind 3 =
// "average" (GWKAverageOrMode: every source pixel the destination pixel's footprint touches — the box spanned by its
// transformed top-left and bottom-right corners — weighted by the covered fraction along each axis, nodata skipped per
// band).  A warp takes 32 consecutive destination pixels: lane = pixel for the fp64 transform, then the lanes sweep the
// bands of one pixel after the other (coalesced records); cubes of few bands keep lane = pixel throughout.
struct PointBox {
    int x0, x1, y0, y1;         // source pixels [x0, x1) x [y0, y1); empty: x1 <= x0
    double xmin, xmax, ymin, ymax;
};

__device__ __forceinline__ PointBox point_box(const WarpParams& P, long long r, long long c) {
    PointBox b;
    b.x0 = b.y0 = 0;
    b.x1 = b.y1 = 0;
    b.xmin = b.xmax = b.ymin = b.ymax = 0.0;
    if (P.kind == 0) {
        double px, py;
        dst_to_src(P, (double)c + 0.5, (double)r + 0.5, px, py);
        if (!(px >= 0.0 && py >= 0.0 && px <= (double)P.Ws && py <= (double)P.Hs)) return b;     // NaN lands here too
        long long ix = (long long)floor(px + 1e-10), iy = (long long)floor(py + 1e-10);
        if (ix == P.Ws) --ix;
        if (iy == P.Hs) --iy;
        b.x0 = (int)ix, b.x1 = (int)ix + 1, b.y0 = (int)iy, b.y1 = (int)iy + 1;
        return b;
    }
    double ax, ay, bx, by;
    dst_to_src(P, (double)c, (double)r, ax, ay);
    dst_to_src(P, (double)c + 1.0, (double)r + 1.0, bx, by);
    if (!(ax == ax && ay == ay && bx == bx && by == by)) return b;
    double xmin = fmin(ax, bx), xmax = fmax(ax, bx), ymin = fmin(ay, by), ymax = fmax(ay, by);
    if (xmax <= 0.0 || ymax <= 0.0 || xmin >= (double)P.Ws || ymin >= (double)P.Hs) return b;
    xmin = fmax(xmin, 0.0), ymin = fmax(ymin, 0.0);                   // the footprint clipped to the source
    xmax = fmin(xmax, (double)P.Ws), ymax = fmin(ymax, (double)P.Hs);
    long long x0 = (long long)floor(xmin + 1e-10), x1 = (long long)ceil(xmax - 1e-10);
    long long y0 = (long long)floor(ymin + 1e-10), y1 = (long long)ceil(ymax - 1e-10);
    if (x0 == x1 && x1 < P.Ws) ++x1;
    if (y0 == y1 && y1 < P.Hs) ++y1;
    b.x0 = (int)x0, b.x1 = (int)x1, b.y0 = (int)y0, b.y1 = (int)y1;
    b.xmin = xmin, b.xmax = xmax, b.ymin = ymin, b.ymax = ymax;
    return b;
}

__device__ __forceinline__ double cover(int i, int i0, int i1, double lo, double hi) {   // COMPUTE_WEIGHT of gdalwarpkernel.cpp
    if (i == i0) return i0 + 1 == i1 ? 1.0 : 1.0 - (lo - (double)i0);
    if (i + 1 == i1) return 1.0 - ((double)i1 - hi);
    return 1.0;
}

__device__ __forceinline__ float point_value(const WarpParams& P, const PointBox& b, int band) {
    if (b.x1 <= b.x0 || b.y1 <= b.y0) return P.dst_nodata;
    if (P.kind == 0) {
        const float v = __ldg(P.src + ((long long)b.y0 * P.Ws + b.x0) * P.src_pix_stride + band);
        return (P.has_nodata && v == P.nodata) ? P.dst_nodata : v;
    }
    double tot = 0.0, wsum = 0.0;
    for (int y = b.y0; y < b.y1; ++y) {
        const double wy = cover(y, b.y0, b.y1, b.ymin, b.ymax);
        const float* row = P.src + ((long long)y * P.Ws) * P.src_pix_stride + band;
        for (int x = b.x0; x < b.x1; ++x) {
            const float v = __ldg(row + (long long)x * P.src_pix_stride);
            if (P.has_nodata && v == P.nodata) continue;
            const double w = wy * cover(x, b.x0, b.x1, b.xmin, b.xmax);
            tot += (double)v * w;
            wsum += w;
        }
    }
    return wsum > 0.0 ? (float)(tot / wsum) : P.dst_nodata;
}

__global__ void __launch_bounds__(256) warp_point_kernel(const WarpParams P) {
    const long long n = P.Hd * P.Wd;
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long base = warp * 32; base < n; base += nwarps * 32) {
        const long long o = base + lane;
        PointBox mine;
        mine.x0 = mine.x1 = mine.y0 = mine.y1 = 0;
        mine.xmin = mine.xmax = mine.ymin = mine.ymax = 0.0;
        if (o < n) mine = point_box(P, o / P.Wd, o % P.Wd);
        if (P.bands < 16) {                       // few bands: lane = pixel
            if (o < n)
                for (int b = 0; b < P.bands; ++b) P.dst[o * P.dst_pix_stride + b] = point_value(P, mine, b);
            continue;
        }
        const int npx = n - base < 32 ? (int)(n - base) : 32;
        for (int i = 0; i < npx; ++i) {           // lanes across the bands of pixel base + i
            PointBox b;
            b.x0 = __shfl_sync(0xffffffffu, mine.x0, i), b.x1 = __shfl_sync(0xffffffffu, mine.x1, i);
            b.y0 = __shfl_sync(0xffffffffu, mine.y0, i), b.y1 = __shfl_sync(0xffffffffu, mine.y1, i);
            b.xmin = __shfl_sync(0xffffffffu, mine.xmin, i), b.xmax = __shfl_sync(0xffffffffu, mine.xmax, i);
            b.ymin = __shfl_sync(0xffffffffu, mine.ymin, i), b.ymax = __shfl_sync(0xffffffffu, mine.ymax, i);
            float* out = P.dst + (base + i) * P.dst_pix_stride;
            for (int band = lane; band < P.bands; band += 32) out[band] = point_value(P, b, band);
        }
    }
}

// bands b .. b+3 of one spectrum, 4-byte loads unless the records are 16-byte aligned
template <bool SRC_VEC>
__device__ __forceinline__ float4 load_group_raw(const float* __restrict__ rec, int b, int bands, bool act) {
    // bands b .. b+3 of one spectrum (words beyond `bands`: record padding with SRC_VEC, 0 otherwise)
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!act) return v;
    if (SRC_VEC) {
        v = __ldg(reinterpret_cast<const float4*>(rec + b));
    } else {
        v.x = __ldg(rec + b);
        if (b + 1 < bands) v.y = __ldg(rec + b + 1);
        if (b + 2 < bands) v.z = __ldg(rec + b + 2);
        if (b + 3 < bands) v.w = __ldg(rec + b + 3);
    }
    return v;
}

// words beyond `bands` take the value of band b, so that they never change what the lane sees of the nodata pattern
__device__ __forceinline__ float4 pad_fix(float4 v, int b, int bands) {
    if (b + 1 >= bands) v.y = v.x;
    if (b + 2 >= bands) v.z = v.x;
    if (b + 3 >= bands) v.w = v.x;
    return v;
}

// ---------------------------------------------------------------------------- lane-per-pixel variant
// Lanes across DESTINATION PIXELS instead of bands.  A CTA owns a 32 x LROWS tile of the destination and walks the
// spectrum in groups of 32 bands (8 float4 "quads"); a thread owns one pixel of the tile for the whole tile: its window
// origin, its separable weights (registers, fully unrolled NT x NT window) and its weight sum are computed ONCE and
// serve every band of the pixel — in the band-per-lane kernels this design replaced, that per-pixel work was redone by
// a whole warp for every pixel and band group, and it dominated them.  Per group the box of the tile's windows is
// staged in shared memory TRANSPOSED ([quad][pixel], odd pitch): the coalesced global reads (lanes across the quads of
// two source pixels) become conflict-free shared-memory writes, and the taps of 32 neighbouring destination pixels — 32
// nearly consecutive source pixels of one quad — are conflict-free 16-byte reads.  The box covers the windows UNCLIPPED
// (pixels outside the source are staged as zeros and carry zero weight), so tap addresses are base + j * bw + k with k
// an immediate.  Groups whose box holds no nodata and no non-finite value take a lean loop (5 instructions per tap and
// quad); the others select weights and values per element.  Three CTAs per SM (single buffer each): staging of one
// overlaps resampling of another.
constexpr int LROWS = 8;            // destination tile: LCOLS x LROWS pixels, one per thread and quad half
constexpr int LCOLS = 16;
constexpr int LQ = 8;               // quads (float4) per band group: 32 bands
constexpr int LBOX = 480;           // staged source pixels per tile (pitch LBOX + 1, odd): 8 * 481 * 16 B = 61.6 KB, 3 CTAs per SM
constexpr int LPITCH = LBOX + 1;

template <int NT, bool DST_VEC>
__global__ void __launch_bounds__(256, 3) warp_lane_kernel(const WarpParams P, const int src_vec) {
    extern __shared__ __align__(16) float4 lbox[];           // [LQ][LPITCH]
    __shared__ int s_mm[4];
    __shared__ float s_wy[NT][256];                          // row weights per thread (the row loop stays rolled)
    __shared__ unsigned int s_pix[LBOX];                     // source pixel index of every box pixel, 0xffffffff outside
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    // a quarter-warp (the unit of a 16-byte shared-memory access) = 8 ROWS of one destination column: their taps sit
    // ~one box row apart, and the box pitch is odd, so the 8 addresses fall into 8 different 16-byte bank groups
    // (neighbouring columns would be 1.2 source pixels apart at the granule's x-scale: two of eight always collide)
    const int prow = lane & 7;                               // my pixel: row prow, column pcol of the tile
    const int pcol = (wib & 3) * 4 + (lane >> 3);
    const int qhalf = wib >> 2;                              // 8 warps = 4 column groups x 2 halves of the group's quads
    constexpr int R = NT / 2;
    const long long tiles_x = (P.Wd + LCOLS - 1) / LCOLS, tiles_y = (P.Hd + LROWS - 1) / LROWS, ntiles = tiles_x * tiles_y;
    const int nvec = (P.bands + 3) >> 2;
    const int ngroups = (nvec + LQ - 1) / LQ;
    const float nd = P.nodata, dnd = P.dst_nodata;
    const bool has_nd = P.has_nodata != 0;
    const long long stride = P.src_pix_stride;

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long ty = tile / tiles_x, tx = tile - ty * tiles_x;
        const long long r = ty * LROWS + prow, c = tx * LCOLS + pcol;
        // ---- my pixel: source coordinates, window origin, weights (once per tile)
        double px = -1.0, py = -1.0;
        if (r < P.Hd && c < P.Wd) {
            const double2 xy = __ldg(reinterpret_cast<const double2*>(P.coords) + (r * P.Wd + c));
            px = xy.x;
            py = xy.y;
        }
        const bool inside = px >= 0.0 && px < (double)P.Ws && py >= 0.0 && py < (double)P.Hs;
        const double fxp = floor(px - 0.5), fyp = floor(py - 0.5);
        const int wx0 = inside ? (int)fxp + 1 - R : 0, wy0 = inside ? (int)fyp + 1 - R : 0;     // first tap of my window
        float wx[NT], wy[NT];
        float wsum_all = 0.f;
        {
            const double ddx = px - 0.5 - fxp, ddy = py - 0.5 - fyp;
            float sx = 0.f, sy = 0.f;
#pragma unroll
            for (int k = 0; k < NT; ++k) {
                // tap k of the NT-wide register window is tap k + P.rx - R of the filter (NT >= 2 * radius)
                const int tk = k + 1 - R;
                const bool inx = inside && tk >= 1 - P.rx && tk <= P.rx && wx0 + k >= 0 && wx0 + k < P.Ws;
                const bool iny = inside && tk >= 1 - P.ry && tk <= P.ry && wy0 + k >= 0 && wy0 + k < P.Hs;
                wx[k] = inx ? (float)tap_weight(P.kind, ((double)tk - ddx) * P.fx) : 0.f;
                wy[k] = iny ? (float)tap_weight(P.kind, ((double)tk - ddy) * P.fy) : 0.f;
                sx += wx[k];
                sy += wy[k];
            }
#pragma unroll
            for (int j = 0; j < NT; ++j) {
#pragma unroll
                for (int k = 0; k < NT; ++k) wsum_all += wy[j] * wx[k];
                s_wy[j][tid] = wy[j];       // read back by this thread only
            }
            (void)sx;
            (void)sy;
        }
        // ---- bounding box of the tile's windows (unclipped)
        if (tid < 4) s_mm[tid] = (tid & 1) ? -2147483647 : 2147483647;
        __syncthreads();
        if (qhalf == 0) {
            const unsigned int FULL = 0xffffffffu;
            const int mnx = __reduce_min_sync(FULL, inside ? wx0 : 2147483647), mxx = __reduce_max_sync(FULL, inside ? wx0 : -2147483647);
            const int mny = __reduce_min_sync(FULL, inside ? wy0 : 2147483647), mxy = __reduce_max_sync(FULL, inside ? wy0 : -2147483647);
            if (lane == 0) {
                atomicMin(&s_mm[0], mnx);
                atomicMax(&s_mm[1], mxx);
                atomicMin(&s_mm[2], mny);
                atomicMax(&s_mm[3], mxy);
            }
        }
        __syncthreads();
        const bool any_inside = s_mm[1] >= s_mm[0];
        const int bx0 = s_mm[0], by0 = s_mm[2];
        const int bw = any_inside ? ((s_mm[1] - s_mm[0] + NT) | 1) : 0, bh = any_inside ? s_mm[3] - s_mm[2] + NT : 0;   // odd pitch
        const int nbox = bw * bh;
        const bool staged = any_inside && nbox <= LBOX;
        const int mybase = (wy0 - by0) * bw + (wx0 - bx0);          // my window's first tap inside the box
        // where every box pixel lives in the source (the same for all band groups of the tile): computed once
        if (staged) {
            for (int p = tid; p < nbox; p += 256) {
                const int by = p / bw, bx = p - by * bw;
                const long long yy = (long long)by0 + by, xx = (long long)bx0 + bx;
                s_pix[p] = (yy >= 0 && yy < P.Hs && xx >= 0 && xx < P.Ws) ? (unsigned int)(yy * P.Ws + xx) : 0xffffffffu;
            }
        }
        __syncthreads();
        float* outp = P.dst + (r * P.Wd + c) * P.dst_pix_stride;

        for (int g = 0; g < ngroups; ++g) {
            const int q0 = g * LQ;
            // ---- stage the box: item i = pixel * LQ + quad; out-of-source pixels and quads beyond the spectrum are zeros
            bool dirty = false, notfill = false;
            if (staged) {
                // thread -> quad (tid & 7) of pixels (tid >> 3), + 32, ...: a warp reads 4 pixels x 128 contiguous bytes and
                // writes 8 runs of 4 consecutive slots (pitch odd: conflict-free); no division, one running box position
                const int q = tid & (LQ - 1);
                const int b = (q0 + q) * 4;
                const bool qok = b < P.bands;
                float4* dstq = lbox + q * LPITCH;
                constexpr int SU = 4;
                for (int p0 = tid >> 3; p0 < nbox; p0 += 32 * SU) {
                    float4 v[SU];
                    bool live[SU];
#pragma unroll
                    for (int u = 0; u < SU; ++u) {
                        const int p = p0 + 32 * u;
                        const unsigned int pix = p < nbox ? s_pix[p] : 0xffffffffu;
                        live[u] = qok && pix != 0xffffffffu;
                        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (live[u]) {
                            const float* rec = P.src + (long long)pix * stride + b;
                            if (src_vec) {
                                v[u] = __ldg(reinterpret_cast<const float4*>(rec));
                            } else {
                                v[u].x = __ldg(rec);
                                if (b + 1 < P.bands) v[u].y = __ldg(rec + 1);
                                if (b + 2 < P.bands) v[u].z = __ldg(rec + 2);
                                if (b + 3 < P.bands) v[u].w = __ldg(rec + 3);
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < SU; ++u) {
                        const int p = p0 + 32 * u;
                        if (p >= nbox) break;
                        float4 x = v[u];
                        if (live[u]) {
                            x = pad_fix(x, b, P.bands);
                            const float z = fmaf(x.x, 0.f, fmaf(x.y, 0.f, fmaf(x.z, 0.f, x.w * 0.f)));
                            dirty = dirty || !(z == 0.f) || (has_nd && (x.x == nd || x.y == nd || x.z == nd || x.w == nd));
                            notfill = notfill || !has_nd || !(x.x == nd && x.y == nd && x.z == nd && x.w == nd);
                        }
                        dstq[p] = x;
                    }
                }
            }
            const bool clean = __syncthreads_or(dirty) == 0;
            // a group whose box holds nothing but nodata (the tile lies outside the swath): every weight sum is 0
            const bool allfill = staged && !clean && __syncthreads_or(notfill) == 0;
            // ---- resample my pixel for my half of the group's quads
            auto store_quad = [&](int b, const float4& o) {
                if (!(r < P.Hd && c < P.Wd) || b >= P.bands) return;
                if (DST_VEC) {
                    __stcs(reinterpret_cast<float4*>(outp + b), o);
                } else {
                    __stcs(outp + b, o.x);
                    if (b + 1 < P.bands) __stcs(outp + b + 1, o.y);
                    if (b + 2 < P.bands) __stcs(outp + b + 2, o.z);
                    if (b + 3 < P.bands) __stcs(outp + b + 3, o.w);
                }
            };
            const float4 fillq = make_float4(dnd, dnd, dnd, dnd);
            // accumulated weights that cancel below 0.03 amplify the fp32 rounding of this kernel beyond the 1e-5 bar: such
            // (pixel, group) pairs are listed and recomputed in fp64 by warp_exact_kernel (as for warp_quad_kernel)
            bool ill = false;
            if (!inside || allfill) {
                for (int qq = 0; qq < LQ / 2; ++qq) store_quad((q0 + qhalf * (LQ / 2) + qq) * 4, fillq);
            } else if (staged && clean) {
                // lean loop, two quads at a time: one weight product serves eight FMAs, two independent accumulator sets
                const float inv_ok = wsum_all >= 1e-6f ? 1.f : 0.f;
                ill = fabsf(wsum_all) < 0.03f && wsum_all != 0.f;
                for (int qq = 0; qq < LQ / 2; qq += 2) {
                    const int q = qhalf * (LQ / 2) + qq;
                    const float4* wp = lbox + q * LPITCH + mybase;
                    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
#pragma unroll 1
                    for (int j = 0; j < NT; ++j) {
                        const float4* rp = wp + j * bw;
                        const float wyj = s_wy[j][tid];
#pragma unroll
                        for (int k = 0; k < NT; ++k) {
                            const float w = wyj * wx[k];
                            const float4 v = rp[k], u = rp[k + LPITCH];
                            a0 = fmaf(w, v.x, a0);
                            a1 = fmaf(w, v.y, a1);
                            a2 = fmaf(w, v.z, a2);
                            a3 = fmaf(w, v.w, a3);
                            c0 = fmaf(w, u.x, c0);
                            c1 = fmaf(w, u.y, c1);
                            c2 = fmaf(w, u.z, c2);
                            c3 = fmaf(w, u.w, c3);
                        }
                    }
                    float4 o = fillq, o2 = fillq;
                    if (inv_ok != 0.f) {
                        o = make_float4(__fdiv_rn(a0, wsum_all), __fdiv_rn(a1, wsum_all), __fdiv_rn(a2, wsum_all), __fdiv_rn(a3, wsum_all));
                        o2 = make_float4(__fdiv_rn(c0, wsum_all), __fdiv_rn(c1, wsum_all), __fdiv_rn(c2, wsum_all), __fdiv_rn(c3, wsum_all));
                    }
                    store_quad((q0 + q) * 4, o);
                    store_quad((q0 + q + 1) * 4, o2);
                }
            } else {
                for (int qq = 0; qq < LQ / 2; ++qq) {
                    const int q = qhalf * (LQ / 2) + qq;
                    const int b = (q0 + q) * 4;
                    if (b >= P.bands) break;
                    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f;
#pragma unroll 1
                    for (int j = 0; j < NT; ++j) {
                        const float wyj = s_wy[j][tid];
#pragma unroll
                        for (int k = 0; k < NT; ++k) {
                            const float w = wyj * wx[k];
                            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (staged) {
                                v = lbox[q * LPITCH + mybase + j * bw + k];
                            } else if (w != 0.f) {      // box too large for the buffer: the tap from global memory
                                const float* rec = P.src + (((long long)wy0 + j) * P.Ws + (wx0 + k)) * stride + b;
                                if (src_vec) {
                                    v = __ldg(reinterpret_cast<const float4*>(rec));
                                } else {
                                    v.x = __ldg(rec);
                                    if (b + 1 < P.bands) v.y = __ldg(rec + 1);
                                    if (b + 2 < P.bands) v.z = __ldg(rec + 2);
                                    if (b + 3 < P.bands) v.w = __ldg(rec + 3);
                                }
                                v = pad_fix(v, b, P.bands);
                            }
                            // a zero weight contributes nothing (not even a NaN); nodata is skipped per element
                            const bool z = w == 0.f;
                            const bool s0 = z || (has_nd && v.x == nd), s1 = z || (has_nd && v.y == nd);
                            const bool s2 = z || (has_nd && v.z == nd), s3 = z || (has_nd && v.w == nd);
                            a0 = fmaf(s0 ? 0.f : w, s0 ? 0.f : v.x, a0);
                            a1 = fmaf(s1 ? 0.f : w, s1 ? 0.f : v.y, a1);
                            a2 = fmaf(s2 ? 0.f : w, s2 ? 0.f : v.z, a2);
                            a3 = fmaf(s3 ? 0.f : w, s3 ? 0.f : v.w, a3);
                            m0 += s0 ? 0.f : w;
                            m1 += s1 ? 0.f : w;
                            m2 += s2 ? 0.f : w;
                            m3 += s3 ? 0.f : w;
                        }
                    }
                    float4 o;
                    o.x = m0 >= 1e-6f ? __fdiv_rn(a0, m0) : dnd;
                    o.y = m1 >= 1e-6f ? __fdiv_rn(a1, m1) : dnd;
                    o.z = m2 >= 1e-6f ? __fdiv_rn(a2, m2) : dnd;
                    o.w = m3 >= 1e-6f ? __fdiv_rn(a3, m3) : dnd;
                    store_quad(b, o);
                    const float mm = fminf(fminf(fabsf(m0), fabsf(m1)), fminf(fabsf(m2), fabsf(m3)));
                    ill = ill || (mm < 0.03f && (m0 != 0.f || m1 != 0.f || m2 != 0.f || m3 != 0.f));
                }
            }
            if (ill && r < P.Hd && c < P.Wd) {
                const unsigned int pos = atomicAdd(P.redo_count, 1u);
                if (pos < P.redo_cap) P.redo_list[pos] = ((unsigned long long)(r * P.Wd + c) << 8) | (unsigned int)g;
            }
            __syncthreads();            // the next group overwrites the box
        }
    }
}

// ---------------------------------------------------------------------------- 2 x 2 block kernel, TMA-staged (default)
// What the r1 / r2 profiles of the lane-per-pixel kernels showed (profiles/r2/warp_notes.md): (1) the tap loops are
// bound by SHARED-MEMORY BANDWIDTH — one 16-byte read per tap, quad and pixel (360 M wavefronts); (2) staging through
// LDG / cp.async is bound by the number of outstanding L1 misses an SM can track, not by HBM or L2 (8 B/clk per SM,
// DRAM 11 % busy): with few taps (bilinear) the kernel still took 70 % of the cubic time.  This kernel removes both:
//   * STAGING BY TMA: one cp.async.bulk.tensor.3d per band group brings the whole box {32 bands, BW pixels, BH rows}
//     of the tile's windows into shared memory (SASS UTMALDG), zero-filling everything outside the source and beyond
//     the last band — no address arithmetic, no registers, no L1 miss tracking; two buffers, the next group in flight
//     while this one is resampled;
//   * 2 x 2 DESTINATION PIXELS PER 8-LANE GROUP: the four windows overlap (neighbours start 1 / scale source pixels
//     apart), so the block reads the UNION frame once — at most (NTX + 2) x (NTY + 2) taps, on average 7.2 x 7.1 = 51
//     reads for four pixels instead of 4 x 36 — and every value read feeds all four.  Each pixel's x weights are held
//     in FRAME coordinates (zero outside its own window) so the loops are static; frame columns / rows beyond the
//     block's actual union are predicated off per lane group and cost no shared-memory bandwidth.  EXACT windows
//     (NTX x NTY = 2 rx x 2 ry, not a square register window), separable evaluation with packed FMAs (fma.rn.f32x2,
//     scalar weight x two samples): per frame row t = sum_k wx[k] * v[k], then acc += wy[j] * t;
//   * lane = QUAD (4 bands) of a block: the 8 lanes of a quarter-warp read the 8 quads of ONE source pixel — 128
//     contiguous bytes, conflict-free without padding or swizzle in the pixel-major layout TMA writes — and store 128
//     contiguous bytes of one destination pixel.
// Boxes that hold a nodata or a non-finite sample take the exact per-element loop over the same frame (nodata skipped
// per band, zero weights contribute nothing); a block whose union does not fit the frame makes its tile run the four
// pixels one after the other through the same code (frame = the pixel's own window); a tile whose box exceeds the
// TMA box reads its taps from global memory.  Needs 16-byte aligned records on both sides; other cubes take
// warp_lane_kernel.
constexpr int QCOLS = 16, QROWS = 8;        // destination tile: 8 x 4 blocks of 2 x 2 pixels, 8 lanes (quads) per block

__device__ __forceinline__ unsigned long long pack2(float a, float b) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long p, float& a, float& b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(p));
}
__device__ __forceinline__ void fma2(unsigned long long& acc, unsigned long long a, unsigned long long b) {   // acc += a * b
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// 16-byte shared-memory load from a 32-bit shared address + immediate offset (one live address register per tap row)
template <int OFF>
__device__ __forceinline__ void lds128(unsigned int addr, unsigned long long& lo, unsigned long long& hi) {
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2+%3];" : "=l"(lo), "=l"(hi) : "r"(addr), "n"(OFF));
}
__device__ __forceinline__ float4 lds128f(unsigned int addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// one box {32 bands from band b0, BW pixels from x0, BH rows from y0} -> shared memory; completes on the mbarrier
__device__ __forceinline__ void tma_load_box(void* dst_smem, const void* tmap, int b0, int x0, int y0, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(dst_smem)),
        "l"(tmap), "r"(b0), "r"(x0), "r"(y0), "r"(smem_u32(bar))
        : "memory");
}

struct QuadGeo {
    int BW, BH;                 // TMA box (pixels, rows); the shared-memory row pitch is BW * 128 bytes
};

// One destination pixel, one quad, exactly: fp64 accumulation of the weighted samples and of the weights (GDAL
// accumulates in double), nodata skipped per band, zero weights contribute nothing (not even a NaN); taps from global
// memory when the box was not staged.  Deliberately NOT inlined and fed from shared memory only (frame-coordinate
// weights wx[ncols], wy[nrows * 4] strided by 4): the mixed / non-finite groups use it for every pixel, the fast loops
// for the few pixels whose weight sum is small (taps lost to the source's border or to fill pixels — the quotient of
// two nearly cancelled fp32 sums is not accurate to 1e-5 below a weight sum of ~0.05); keeping it out of line keeps
// its registers out of the fast loops.
struct ExactArgs {
    const float* src;           // global taps (box not staged)
    long long Hs, Ws, stride;
    unsigned int tap0;          // shared address of frame tap (0, 0), my quad; 0 = not staged
    unsigned int rowpitch;      // bytes between frame rows in shared memory
    unsigned int wx_s, wy_s;    // shared addresses: wx[k] (4-byte stride), wy[j] (16-byte stride)
    int ax, ay, ncols, nrows;   // frame origin in the source, extent
    int b, bands, has_nd, inside;
    float nd, dnd;
};

// `ill`: some band's accumulated weight is small (|m| < 0.03): its quotient amplifies the last bit of the fp32 weight
// factors used here by 1 / m — the caller lists the pixel for warp_exact_kernel, which forms the weights as the oracle does.
__device__ __noinline__ float4 warp_exact_pixel(const ExactArgs A, bool& ill) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;
    for (int j = 0; j < A.nrows; ++j) {
        float wyj;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(wyj) : "r"(A.wy_s + (unsigned int)j * 16u));
        if (wyj == 0.f) continue;
        for (int k = 0; k < A.ncols; ++k) {
            float wxk;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(wxk) : "r"(A.wx_s + (unsigned int)k * 4u));
            const double w = (double)wyj * (double)wxk;
            if (w == 0.0) continue;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (A.tap0) {
                v = lds128f(A.tap0 + (unsigned int)j * A.rowpitch + (unsigned int)k * 128u);
            } else {
                const long long yy = (long long)A.ay + j, xx = (long long)A.ax + k;
                if (yy >= 0 && yy < A.Hs && xx >= 0 && xx < A.Ws)
                    v = __ldg(reinterpret_cast<const float4*>(A.src + (yy * A.Ws + xx) * A.stride + A.b));
            }
            v = pad_fix(v, A.b, A.bands);
            if (!(A.has_nd && v.x == A.nd)) { a0 = fma(w, (double)v.x, a0); m0 += w; }
            if (!(A.has_nd && v.y == A.nd)) { a1 = fma(w, (double)v.y, a1); m1 += w; }
            if (!(A.has_nd && v.z == A.nd)) { a2 = fma(w, (double)v.z, a2); m2 += w; }
            if (!(A.has_nd && v.w == A.nd)) { a3 = fma(w, (double)v.w, a3); m3 += w; }
        }
    }
    float4 o;
    o.x = (A.inside && m0 >= 1e-6) ? (float)(a0 / m0) : A.dnd;
    o.y = (A.inside && m1 >= 1e-6) ? (float)(a1 / m1) : A.dnd;
    o.z = (A.inside && m2 >= 1e-6) ? (float)(a2 / m2) : A.dnd;
    o.w = (A.inside && m3 >= 1e-6) ? (float)(a3 / m3) : A.dnd;
    const double ms = fmin(fmin(fabs(m0), fabs(m1)), fmin(fabs(m2), fabs(m3)));
    ill = A.inside && ms < 0.03 && (m0 != 0.0 || m1 != 0.0 || m2 != 0.0 || m3 != 0.0);
    return o;
}

// The exact pass: one lane per (destination pixel, quad of 4 bands), fp64 accumulation (GDAL accumulates in double) straight
// from global memory; any radius up to MAX_TAPS / 2, any record alignment, 64-bit indices.  Two modes:
//   * the fix-up (dense = false): the (pixel, band group) entries the quad and lane kernels listed because their weight sum
//     came out small (taps lost to fill pixels or to the source's border: the quotient of two nearly cancelled fp32 sums is
//     not accurate to 1e-5 below a weight sum of ~0.03), 8 lanes per entry.  A ring a fraction of a pixel wide around
//     the swath: a few thousand entries per granule;
//   * dense: every (pixel, quad) of the destination — filters wider than the fast kernels hold (radius > 4) and sources of
//     2^32 pixels or more.
__global__ void __launch_bounds__(256) warp_exact_kernel(const WarpParams P, const bool dense) {
    const int nvec = (P.bands + 3) >> 2;
    const long long n = dense ? P.Hd * P.Wd * nvec : (long long)LQ * (*P.redo_count < P.redo_cap ? *P.redo_count : P.redo_cap);
    const bool src_vec = (P.src_pix_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(P.src) & 15) == 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        long long pix;
        int qi;
        if (dense) {
            pix = i / nvec;
            qi = (int)(i - pix * nvec);
        } else {
            const unsigned long long ent = P.redo_list[i / LQ];
            pix = (long long)(ent >> 8);
            qi = (int)(ent & 0xffu) * LQ + (int)(i % LQ);
            if (qi >= nvec) continue;
        }
        const int b = qi * 4;
        const double2 xy = __ldg(reinterpret_cast<const double2*>(P.coords) + pix);
        const double px = xy.x, py = xy.y;
        float4 o = make_float4(P.dst_nodata, P.dst_nodata, P.dst_nodata, P.dst_nodata);
        if (px >= 0.0 && px < (double)P.Ws && py >= 0.0 && py < (double)P.Hs) {     // listed entries always are
            const double fxp = floor(px - 0.5), fyp = floor(py - 0.5);
            const long long x0 = (long long)fxp + 1 - P.rx, y0 = (long long)fyp + 1 - P.ry;
            const double ddx = px - 0.5 - fxp, ddy = py - 0.5 - fyp;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;
            for (int j = 0; j < 2 * P.ry; ++j) {
                const long long yy = y0 + j;
                if (yy < 0 || yy >= P.Hs) continue;
                const double wy = tap_weight(P.kind, ((double)(j + 1 - P.ry) - ddy) * P.fy);
                if (wy == 0.0) continue;
                for (int k = 0; k < 2 * P.rx; ++k) {
                    const long long xx = x0 + k;
                    if (xx < 0 || xx >= P.Ws) continue;
                    // ONE rounding to fp32, of the product of the fp64 factors: the convention of oracle/warp.py.  (Rounding
                    // the factors separately, as the fast loops do, moves a quotient whose weights cancel to 1e-4 by 1e-3.)
                    const double w = (double)(float)(wy * tap_weight(P.kind, ((double)(k + 1 - P.rx) - ddx) * P.fx));
                    if (w == 0.0) continue;
                    const float* rec = P.src + (yy * P.Ws + xx) * P.src_pix_stride;
                    const float4 v = pad_fix(src_vec ? load_group_raw<true>(rec, b, P.bands, true) : load_group_raw<false>(rec, b, P.bands, true),
                                             b, P.bands);
                    const bool hn = P.has_nodata != 0;
                    if (!(hn && v.x == P.nodata)) { a0 = fma(w, (double)v.x, a0); m0 += w; }
                    if (!(hn && v.y == P.nodata)) { a1 = fma(w, (double)v.y, a1); m1 += w; }
                    if (!(hn && v.z == P.nodata)) { a2 = fma(w, (double)v.z, a2); m2 += w; }
                    if (!(hn && v.w == P.nodata)) { a3 = fma(w, (double)v.w, a3); m3 += w; }
                }
            }
            if (m0 >= 1e-6) o.x = (float)(a0 / m0);
            if (m1 >= 1e-6) o.y = (float)(a1 / m1);
            if (m2 >= 1e-6) o.z = (float)(a2 / m2);
            if (m3 >= 1e-6) o.w = (float)(a3 / m3);
        }
        float* op = P.dst + pix * P.dst_pix_stride + b;
        if (((reinterpret_cast<uintptr_t>(op) & 15) == 0) && b + 3 < P.dst_pix_stride) {
            *reinterpret_cast<float4*>(op) = o;
        } else {
            op[0] = o.x;
            if (b + 1 < P.bands) op[1] = o.y;
            if (b + 2 < P.bands) op[2] = o.z;
            if (b + 3 < P.bands) op[3] = o.w;
        }
    }
}

template <int NTX, int NTY, bool DST_VEC>
__global__ void __launch_bounds__(256, 2) warp_quad_kernel(const __grid_constant__ CUtensorMap tmap, const WarpParams P,
                                                           const QuadGeo G) {
    constexpr int FW = NTX + 2, FH = NTY + 2;                // frame of a 2 x 2 block
    constexpr int RX = NTX / 2, RY = NTY / 2;
    constexpr unsigned int FULL = 0xffffffffu;
    extern __shared__ __align__(128) unsigned char qsmem[];  // [2 buffers][BH][BW][32 floats]
    __shared__ __align__(8) uint64_t s_full[2];
    __shared__ int s_mm[4];
    __shared__ __align__(16) float s_wy[32][FH][4];          // per block and frame row: the four pixels' row weights
    __shared__ unsigned char s_cls[1024];                    // per box pixel (dirty groups only): 0 clean, 1 fill, 2 mixed
    __shared__ float s_wx[32][4][FW];                        // per block and pixel: column weights in frame coordinates (exact path)
    const int tid = threadIdx.x, lane = tid & 31;
    const int q = tid & 7;                                   // my quad of the band group
    const int blk = tid >> 3;                                // my block: block column blk & 7, block row blk >> 3
    const int sub = lane & ~7;                               // first lane of my 8-lane group
    const long long tiles_x = (P.Wd + QCOLS - 1) / QCOLS, tiles_y = (P.Hd + QROWS - 1) / QROWS, ntiles = tiles_x * tiles_y;
    const int nvec = (P.bands + 3) >> 2;
    const int ngroups = (nvec + LQ - 1) / LQ;
    const float nd = P.nodata, dnd = P.dst_nodata;
    const bool has_nd = P.has_nodata != 0;
    const long long stride = P.src_pix_stride;
    const unsigned int buf_bytes = (unsigned int)(G.BW * G.BH) * 128u;
    const unsigned int rowpitch = (unsigned int)G.BW * 128u;
    const unsigned int qs = smem_u32(qsmem);
    const unsigned int wy_s = smem_u32(&s_wy[blk][0][0]);
    if (tid == 0) {
        mbar_init(&s_full[0], 1);
        mbar_init(&s_full[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    unsigned int uses0 = 0, uses1 = 0;                       // completed phases of the two full barriers (uniform)

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long ty = tile / tiles_x, tx = tile - ty * tiles_x;
        const long long r0 = ty * QROWS + 2 * (blk >> 3), c0 = tx * QCOLS + 2 * (blk & 7);   // my block's first pixel
        // ---- set-up, shared by the 8 lanes of the block: lane p (< 4) owns pixel p's column axis, lane 4 + p its row
        //      axis (pixel p = (row r0 + (p >> 1), column c0 + (p & 1)))
        const int mp = q & 3;
        const long long mr = r0 + (mp >> 1), mc = c0 + (mp & 1);
        const bool mexists = mr < P.Hd && mc < P.Wd;
        double px = -1.0, py = -1.0;
        if (mexists) {
            const double2 xy = __ldg(reinterpret_cast<const double2*>(P.coords) + (mr * P.Wd + mc));
            px = xy.x;
            py = xy.y;
        }
        const bool mins = px >= 0.0 && px < (double)P.Ws && py >= 0.0 && py < (double)P.Hs;
        const bool xaxis = q < 4;
        const double cc = xaxis ? px : py;
        const double fl = floor(cc - 0.5);
        const int w0 = mins ? (int)fl + 1 - (xaxis ? RX : RY) : 0;        // first tap of my pixel's window on my axis
        constexpr int NTM = NTX > NTY ? NTX : NTY;
        float wo[NTM];                                                     // own-window weights on my axis
        float wsum = 0.f;
        {
            const double dd = cc - 0.5 - fl, f = xaxis ? P.fx : P.fy;
            const long long lim = xaxis ? P.Ws : P.Hs;
            const int nt = xaxis ? NTX : NTY, rad = xaxis ? RX : RY;
#pragma unroll
            for (int k = 0; k < NTM; ++k) {
                const bool in = mins && k < nt && w0 + k >= 0 && w0 + k < lim;
                wo[k] = in ? (float)tap_weight(P.kind, ((double)(k + 1 - rad) - dd) * f) : 0.f;
                wsum += wo[k];
            }
        }
        // the block's four window origins, inside flags, normalisation
        int wx0[4], wy0[4];
        float winv[4];
        const unsigned int insb = (__ballot_sync(FULL, mins) >> sub) & 0xfu;          // bit p: pixel p inside the source
        const unsigned int exb = (__ballot_sync(FULL, mexists) >> sub) & 0xfu;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            wx0[p] = __shfl_sync(FULL, w0, sub + p);
            wy0[p] = __shfl_sync(FULL, w0, sub + 4 + p);
            const float sx = __shfl_sync(FULL, wsum, sub + p), sy = __shfl_sync(FULL, wsum, sub + 4 + p);
            const float ws = sx * sy;
            winv[p] = (((insb >> p) & 1u) && ws >= 1e-6f) ? 1.f / ws : 0.f;           // 0: the pixel is left at dst_nodata
        }
        // ---- the block's frame: anchored at the smallest origin of the windows that are inside; does the union fit?
        int fx0 = 2147483647, fy0 = 2147483647, mxx = -2147483647, mxy = -2147483647;
#pragma unroll
        for (int p = 0; p < 4; ++p)
            if ((insb >> p) & 1u) {
                fx0 = wx0[p] < fx0 ? wx0[p] : fx0;
                fy0 = wy0[p] < fy0 ? wy0[p] : fy0;
                mxx = wx0[p] > mxx ? wx0[p] : mxx;
                mxy = wy0[p] > mxy ? wy0[p] : mxy;
            }
        const bool misfit = insb != 0u && (mxx - fx0 + NTX > FW || mxy - fy0 + NTY > FH);
        // ---- bounding box of the tile's windows (unclipped)
        if (tid < 4) s_mm[tid] = (tid & 1) ? -2147483647 : 2147483647;
        __syncthreads();
        {
            const int big = 2147483647;
            const int mnx = __reduce_min_sync(FULL, insb ? fx0 : big), mx2 = __reduce_max_sync(FULL, insb ? mxx : -big);
            const int mny = __reduce_min_sync(FULL, insb ? fy0 : big), my2 = __reduce_max_sync(FULL, insb ? mxy : -big);
            if (lane == 0) {
                atomicMin(&s_mm[0], mnx);
                atomicMax(&s_mm[1], mx2);
                atomicMin(&s_mm[2], mny);
                atomicMax(&s_mm[3], my2);
            }
        }
        const bool solo = __syncthreads_or(misfit) != 0;     // (barrier) some block does not fit: one pixel at a time
        const bool any_inside = s_mm[1] >= s_mm[0];
        const int bx0 = s_mm[0], by0 = s_mm[2];
        const int bw = any_inside ? s_mm[1] - s_mm[0] + NTX : 0, bh = any_inside ? s_mm[3] - s_mm[2] + NTY : 0;
        const bool staged = any_inside && bw <= G.BW && bh <= G.BH;
        // ---- first two band groups on their way (the buffers were released by the closing barrier of the last tile)
        if (staged && tid == 0) {
            mbar_arrive_expect_tx(&s_full[0], buf_bytes);
            tma_load_box(qsmem, &tmap, 0, bx0, by0, &s_full[0]);
            if (ngroups > 1) {
                mbar_arrive_expect_tx(&s_full[1], buf_bytes);
                tma_load_box(qsmem + buf_bytes, &tmap, LQ * 4, bx0, by0, &s_full[1]);
            }
        }
        // ---- weights in frame coordinates (block mode) or own-window coordinates (solo mode: offsets 0)
        float wxf[4][FW];
        {
            const int myoff = solo ? 0 : (mins ? w0 - (xaxis ? fx0 : fy0) : 0);       // my window's offset in the frame: 0, 1, 2
            constexpr int FM = FW > FH ? FW : FH;
            float wf[FM];
#pragma unroll
            for (int k = 0; k < FM; ++k) {
                float w = 0.f;
#pragma unroll
                for (int a = 0; a <= 2; ++a)
                    if (k - a >= 0 && k - a < NTM && myoff == a) w = wo[k - a];
                wf[k] = w;
            }
#pragma unroll
            for (int k = 0; k < FW; ++k)
#pragma unroll
                for (int p = 0; p < 4; ++p) wxf[p][k] = __shfl_sync(FULL, wf[k], sub + p);
            if (!xaxis) {
#pragma unroll
                for (int j = 0; j < FH; ++j) s_wy[blk][j][mp] = wf[j];
            } else {
#pragma unroll
                for (int k = 0; k < FW; ++k) s_wx[blk][mp][k] = wf[k];
            }
            __syncwarp();
        }
        // frame extents actually needed (columns / rows beyond them are predicated off: no shared-memory traffic)
        const int fcols = solo ? NTX : (insb ? mxx - fx0 + NTX : NTX), frows = solo ? NTY : (insb ? mxy - fy0 + NTY : NTY);
        const int rtop_blk = __reduce_max_sync(FULL, frows);                 // rows the warp's row loop runs (all lanes are here)
        float* outp = P.dst + (r0 * P.Wd + c0) * P.dst_pix_stride;          // pixel 0 of my block

        for (int g = 0; g < ngroups; ++g) {
            const int q0 = g * LQ;
            const int buf = g & 1;
            const unsigned int gs = qs + (unsigned int)buf * buf_bytes;       // this group's buffer (shared address)
            bool dirty = false, notfill = false;
            unsigned long long f0 = 0ull, f1 = 0ull;             // running x * 0 of my share of the box (non-finite detector)
            if (staged) {
                mbar_wait(&s_full[buf], (buf ? uses1 : uses0) & 1u);
                if (buf) ++uses1; else ++uses0;
                // classify the box (the bw x bh pixels the windows can touch): 8-lane group i takes pixels i, i + 32, ...
                // of it, lane = quad — 128 contiguous bytes per group and read.  Branch-free, packed: fin += x * 0 (stays 0
                // unless a sample is NaN / Inf); pm = min |prod (x - nd)| (0 iff some sample is the nodata value);
                // sq += (x - nd)^2 (0 iff all are).  Zero-filled pixels / bands are finite and differ from nodata (a nodata
                // of 0 makes them "dirty": the exact loop then skips them by their zero weight or stores nothing for them).
                const unsigned long long nnd = pack2(-nd, -nd);
                unsigned long long s0 = 0ull, s1 = 0ull;
                float pm = 3.0e38f;
                const bool lastg = g == ngroups - 1;                          // only the last group can hold padding / dead quads
                if (!lastg || q < nvec - q0) {
                    const int tailw = P.bands - (q0 + q) * 4;                 // live words of my quad (< 4: the spectrum's last quad)
                    // the part of the box inside the source: columns [xlo, xhi), rows [ylo, yhi) in box coordinates
                    const int xlo = bx0 < 0 ? -bx0 : 0, ylo = by0 < 0 ? -by0 : 0;
                    const int xhi = (long long)bx0 + bw > P.Ws ? (int)(P.Ws - bx0) : bw;
                    const int yhi = (long long)by0 + bh > P.Hs ? (int)(P.Hs - by0) : bh;
                    const int nw = xhi - xlo;
                    if (nw > 0) {
                        // running (row, column) of items blk, blk + 32, ... of the in-source part, no division
                        int bx = xlo + blk, by = ylo;
                        while (bx >= xhi) {
                            bx -= nw;
                            ++by;
                        }
                        unsigned int ad = gs + (unsigned int)(by * G.BW + bx) * 128u + (unsigned int)q * 16u;
                        while (by < yhi) {
                            float4 x = lds128f(ad);
                            if (lastg && tailw < 4) x = pad_fix(x, (q0 + q) * 4, P.bands);
                            const unsigned long long p01 = pack2(x.x, x.y), p23 = pack2(x.z, x.w);
                            fma2(f0, p01, 0ull);
                            fma2(f1, p23, 0ull);
                            const unsigned long long d01 = add2(p01, nnd), d23 = add2(p23, nnd);
                            fma2(s0, d01, d01);
                            fma2(s1, d23, d23);
                            float m0, m1;
                            unpack2(mul2(d01, d23), m0, m1);
                            pm = fminf(pm, fabsf(m0 * m1));
                            bx += 32;
                            ad += 32u * 128u;
                            while (bx >= xhi) {
                                bx -= nw;
                                ++by;
                                ad += rowpitch - (unsigned int)nw * 128u;
                            }
                        }
                    }
                }
                float fa, fb, fc, fd, sa, sb, sc, sd;
                unpack2(f0, fa, fb);
                unpack2(f1, fc, fd);
                unpack2(s0, sa, sb);
                unpack2(s1, sc, sd);
                const bool nonfinite = !((fa + fb) + (fc + fd) == 0.f);
                dirty = nonfinite || (has_nd && pm == 0.f);
                notfill = !has_nd || nonfinite || !((sa + sb) + (sc + sd) == 0.f);
            }
            const bool clean = __syncthreads_or(dirty) == 0;
            const bool allfill = staged && !clean && __syncthreads_or(notfill) == 0;
            // a dirty box (the swath's edge): classify every box pixel — clean, FILL (all bands of the group are nodata: the
            // usual case outside the swath) or mixed.  Without mixed pixels and non-finite samples the group takes the
            // medium loop, which drops fill pixels tap by tap for all bands at once.
            bool fillonly = false;
            if (staged && !clean && !allfill) {
                bool bad = !(G.BW * G.BH <= 1024);
                {
                    float fa, fb, fc, fd;
                    unpack2(f0, fa, fb);
                    unpack2(f1, fc, fd);
                    bad = bad || !((fa + fb) + (fc + fd) == 0.f);
                }
                bad = __any_sync(FULL, bad) != 0;                // warp-uniform: the 8-lane ballots below need whole groups
                if (!bad) {
                    const bool lastg = g == ngroups - 1;
                    const bool deadq = lastg && q >= nvec - q0;
                    const int tailw = P.bands - (q0 + q) * 4;
                    const int xlo = bx0 < 0 ? -bx0 : 0, ylo = by0 < 0 ? -by0 : 0;
                    const int xhi = (long long)bx0 + bw > P.Ws ? (int)(P.Ws - bx0) : bw;
                    const int yhi = (long long)by0 + bh > P.Hs ? (int)(P.Hs - by0) : bh;
                    const int nw = xhi - xlo;
                    const unsigned int gmask = 0xffu << sub;
                    if (nw > 0) {
                        int bx = xlo + blk, by = ylo;
                        while (bx >= xhi) {
                            bx -= nw;
                            ++by;
                        }
                        while (by < yhi) {
                            float4 x = lds128f(gs + (unsigned int)(by * G.BW + bx) * 128u + (unsigned int)q * 16u);
                            if (lastg && tailw < 4) x = pad_fix(x, (q0 + q) * 4, P.bands);
                            const bool anyn = !deadq && (x.x == nd || x.y == nd || x.z == nd || x.w == nd);
                            const bool alln = deadq || (x.x == nd && x.y == nd && x.z == nd && x.w == nd);
                            const unsigned int ba = __ballot_sync(gmask, anyn) & gmask, bl = __ballot_sync(gmask, alln) & gmask;
                            const int cls = ba == 0u ? 0 : (bl == gmask ? 1 : 2);
                            if (q == 0) s_cls[by * G.BW + bx] = (unsigned char)cls;
                            bad = bad || cls == 2;
                            bx += 32;
                            while (bx >= xhi) {
                                bx -= nw;
                                ++by;
                            }
                        }
                    }
                }
                fillonly = __syncthreads_or(bad) == 0;           // (barrier: the class table is visible)
            }
            const int b = (q0 + q) * 4;                                       // my first band
            auto store_px = [&](int p, const float4& o) {
                if (!((exb >> p) & 1u) || b >= P.bands) return;
                float* op = outp + ((long long)(p >> 1) * P.Wd + (p & 1)) * P.dst_pix_stride + b;
                if (DST_VEC) {
                    __stcs(reinterpret_cast<float4*>(op), o);
                } else {
                    __stcs(op, o.x);
                    if (b + 1 < P.bands) __stcs(op + 1, o.y);
                    if (b + 2 < P.bands) __stcs(op + 2, o.z);
                    if (b + 3 < P.bands) __stcs(op + 3, o.w);
                }
            };
            const float4 fillq = make_float4(dnd, dnd, dnd, dnd);
            const int npass = solo ? 4 : 1;
            for (int pass = 0; pass < npass; ++pass) {
                // pixels this pass produces (bit mask), and the frame it reads
                const unsigned int doing = solo ? (1u << pass) : 0xfu;
                const unsigned int live = doing & insb;
                if (allfill || live == 0u) {
#pragma unroll
                    for (int p = 0; p < 4; ++p)
                        if ((doing >> p) & 1u) store_px(p, fillq);
                    continue;
                }
                const int ax = solo ? wx0[pass] : fx0, ay = solo ? wy0[pass] : fy0;      // frame origin in the source
                const int ncols = solo ? NTX : fcols, nrows = solo ? NTY : frows;
                auto exact_px = [&](int p) -> bool {         // see warp_exact_pixel; true: ill-conditioned, to be fixed up
                    if (b >= P.bands) return false;
                    ExactArgs A;
                    A.src = P.src, A.Hs = P.Hs, A.Ws = P.Ws, A.stride = stride;
                    A.tap0 = staged ? gs + (unsigned int)((ay - by0) * G.BW + (ax - bx0)) * 128u + (unsigned int)q * 16u : 0u;
                    A.rowpitch = rowpitch;
                    A.wx_s = smem_u32(&s_wx[blk][p][0]);
                    A.wy_s = wy_s + (unsigned int)p * 4u;
                    A.ax = ax, A.ay = ay, A.ncols = ncols, A.nrows = nrows;
                    A.b = b, A.bands = P.bands, A.has_nd = has_nd ? 1 : 0, A.inside = (int)((insb >> p) & 1u);
                    A.nd = nd, A.dnd = dnd;
                    bool ill = false;
                    store_px(p, warp_exact_pixel(A, ill));
                    return ill;
                };
                auto list_px = [&](int p) {                  // leave (pixel p, this band group) to warp_exact_kernel
                    if (q != 0 || !((exb >> p) & 1u) || P.redo_list == nullptr) return;
                    const unsigned int pos = atomicAdd(P.redo_count, 1u);
                    if (pos < P.redo_cap)
                        P.redo_list[pos] = ((unsigned long long)((r0 + (p >> 1)) * P.Wd + c0 + (p & 1)) << 8) | (unsigned int)g;
                };
                unsigned int redo = 0u;                      // pixels of a mixed / unstaged group: exact_px
                if (staged && clean) {
                    // ---- lean loop.  Rows 0 .. NTY-1 and columns 0 .. NTX-1 of the frame belong to every block; only the
                    //      extra rows / columns are predicated (no warp-wide primitive here: groups without a live pixel
                    //      left above).
                    unsigned int ra = gs + (unsigned int)((ay - by0) * G.BW + (ax - bx0)) * 128u + (unsigned int)q * 16u;
                    unsigned long long acc[4][2] = {{0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}};
                    const int rtop = solo ? NTY : rtop_blk;
#pragma unroll 1
                    for (int j = 0; j < rtop; ++j, ra += rowpitch) {
                        unsigned long long t[4][2] = {{0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}};
                        if (j < NTY || j < nrows) {
                            unsigned long long v0, v1;
#define HSR_TAP(K)                                                                          \
    if ((K) < NTX || ((K) < FW && (K) < ncols)) {                                          \
        lds128<128 * ((K) < FW ? (K) : 0)>(ra, v0, v1);                                    \
        _Pragma("unroll") for (int p = 0; p < 4; ++p) {                                    \
            const unsigned long long w = pack2(wxf[p][(K) < FW ? (K) : 0], wxf[p][(K) < FW ? (K) : 0]); \
            fma2(t[p][0], w, v0);                                                          \
            fma2(t[p][1], w, v1);                                                          \
        }                                                                                  \
    }
                            HSR_TAP(0) HSR_TAP(1) HSR_TAP(2) HSR_TAP(3) HSR_TAP(4)
                            HSR_TAP(5) HSR_TAP(6) HSR_TAP(7) HSR_TAP(8) HSR_TAP(9)
#undef HSR_TAP
                        }
                        const float4 wy = lds128f(wy_s + (unsigned int)j * 16u);
                        const float wyp[4] = {wy.x, wy.y, wy.z, wy.w};
#pragma unroll
                        for (int p = 0; p < 4; ++p) {
                            const float w1 = ((doing >> p) & 1u) ? wyp[p] : 0.f;
                            const unsigned long long w = pack2(w1, w1);
                            fma2(acc[p][0], w, t[p][0]);
                            fma2(acc[p][1], w, t[p][1]);
                        }
                    }
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        if (!((doing >> p) & 1u)) continue;
                        if (winv[p] > 33.f) list_px(p);    // weight sum < 0.03 (taps beyond the source's border)
                        float4 o = fillq;
                        if (winv[p] != 0.f) {
                            const unsigned long long iv = pack2(winv[p], winv[p]);
                            unpack2(mul2(acc[p][0], iv), o.x, o.y);
                            unpack2(mul2(acc[p][1], iv), o.z, o.w);
                        }
                        store_px(p, o);
                    }
                } else if (staged && fillonly) {
                    // ---- medium loop (swath edge): the lean loop, but a FILL pixel (all bands of the group nodata) is skipped
                    //      for the four pixels at once and the weights that remain are summed per pixel
                    unsigned int ra = gs + (unsigned int)((ay - by0) * G.BW + (ax - bx0)) * 128u + (unsigned int)q * 16u;
                    int ci = (ay - by0) * G.BW + (ax - bx0);
                    unsigned long long acc[4][2] = {{0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}};
                    float ms[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
                    for (int j = 0; j < nrows; ++j, ra += rowpitch, ci += G.BW) {
                        unsigned long long t[4][2] = {{0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}, {0ull, 0ull}};
                        float tw[4] = {0.f, 0.f, 0.f, 0.f};
                        // branch-free: the row's class bytes first (independent loads), then every tap with its weights
                        // zeroed where the source pixel is fill (its samples are finite: -9999 * 0 = 0)
                        unsigned int fillmask = 0u;
#pragma unroll
                        for (int k = 0; k < FW; ++k)
                            if (k < ncols && s_cls[ci + k] != 0) fillmask |= 1u << k;
#pragma unroll
                        for (int k = 0; k < FW; ++k) {
                            if (k >= NTX && k >= ncols) break;
                            unsigned long long v0, v1;
                            asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(v0), "=l"(v1) : "r"(ra + (unsigned int)k * 128u));
                            const bool fillpx = (fillmask >> k) & 1u;
#pragma unroll
                            for (int p = 0; p < 4; ++p) {
                                const float w1 = fillpx ? 0.f : wxf[p][k];
                                const unsigned long long w = pack2(w1, w1);
                                fma2(t[p][0], w, v0);
                                fma2(t[p][1], w, v1);
                                tw[p] += w1;
                            }
                        }
                        const float4 wy = lds128f(wy_s + (unsigned int)j * 16u);
                        const float wyp[4] = {wy.x, wy.y, wy.z, wy.w};
#pragma unroll
                        for (int p = 0; p < 4; ++p) {
                            const float w1 = ((doing >> p) & 1u) ? wyp[p] : 0.f;
                            const unsigned long long w = pack2(w1, w1);
                            fma2(acc[p][0], w, t[p][0]);
                            fma2(acc[p][1], w, t[p][1]);
                            ms[p] = fmaf(w1, tw[p], ms[p]);
                        }
                    }
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        if (!((doing >> p) & 1u)) continue;
                        // few valid taps left: fixed up exactly afterwards (a sum <= -1e-3 is clearly below GDAL's 1e-6
                        // threshold, 0 means no valid tap at all: both are nodata without a second look)
                        if (((insb >> p) & 1u) && ms[p] > -1e-3f && ms[p] != 0.f && ms[p] < 0.03f) list_px(p);
                        float4 o = fillq;
                        if (((insb >> p) & 1u) && ms[p] >= 1e-6f) {
                            const float inv = 1.f / ms[p];
                            const unsigned long long iv = pack2(inv, inv);
                            unpack2(mul2(acc[p][0], iv), o.x, o.y);
                            unpack2(mul2(acc[p][1], iv), o.z, o.w);
                        }
                        store_px(p, o);
                    }
                } else {
                    redo = doing;    // mixed / non-finite group (or a box beyond the TMA box): every pixel exactly
                }
                if (redo) {                  // uniform over the 8 lanes of a group only (groups without a live pixel left
                                             // above): the vote is taken under the group's mask
                    const unsigned int gm = 0xffu << sub;
#pragma unroll 1
                    for (int p = 0; p < 4; ++p)
                        if ((redo >> p) & 1u) {
                            const bool ill = exact_px(p);
                            if ((__ballot_sync(gm, ill) & gm) != 0u) list_px(p);
                        }
                }
            }
            __syncthreads();            // everybody is done with this buffer: refill it with the group after next
            if (staged && tid == 0 && g + 2 < ngroups) {
                mbar_arrive_expect_tx(&s_full[buf], buf_bytes);
                tma_load_box(qsmem + (size_t)buf * buf_bytes, &tmap, (g + 2) * LQ * 4, bx0, by0, &s_full[buf]);
            }
        }
    }
}

// ---------------------------------------------------------------------------- K planes, lane per pixel
// hsr_warp_planes_f32: K <= 16 planar images (the pseudo-S2 planes of the SRF pass) resampled with the taps of
// hsr_warp_f32, validity per SOURCE PIXEL (src_valid) instead of per band and value.  One thread per destination pixel
// of a 32 x 8 tile; the K accumulators are fp64 registers (K is a template parameter, every loop over it unrolled), so
// the quotient is formed as warp_exact_kernel forms it and there is no fix-up pass.  Tap weights: the fp32 rounding of
// the fp64 product wy * wx (oracle/warp.py); zero weights, taps outside the source and invalid source pixels skipped.
constexpr int PL_COLS = 32, PL_ROWS = 8;

struct PlaneParams {
    const float* src;
    const uint8_t* src_valid;
    long long Hs, Ws, src_plane_stride;
    const double* coords;
    long long Hd, Wd;
    int kind, rx, ry;
    double fx, fy;
    const float* fill_out;
    int gate_k;
    float gate_gt;
    float* dst;
    long long dst_plane_stride;
    uint8_t* dst_valid;
    uint8_t* fit_mask;
};

template <int K>
__global__ void __launch_bounds__(PL_COLS * PL_ROWS) warp_planes_kernel(const PlaneParams P) {
    const long long c = (long long)blockIdx.x * PL_COLS + threadIdx.x;
    if (c >= P.Wd) return;
    const long long tiles_y = (P.Hd + PL_ROWS - 1) / PL_ROWS;
    for (long long ty = blockIdx.y; ty < tiles_y; ty += gridDim.y) {
        const long long r = ty * PL_ROWS + threadIdx.y;
        if (r >= P.Hd) return;
        const long long o = r * P.Wd + c;
        const double2 xy = __ldg(reinterpret_cast<const double2*>(P.coords) + o);
        const double px = xy.x, py = xy.y;
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.0;
        double ws = 0.0;
        const bool inside = px >= 0.0 && px < (double)P.Ws && py >= 0.0 && py < (double)P.Hs;
        if (inside) {
            const double fxp = floor(px - 0.5), fyp = floor(py - 0.5);
            const long long x0 = (long long)fxp + 1 - P.rx, y0 = (long long)fyp + 1 - P.ry;
            const double ddx = px - 0.5 - fxp, ddy = py - 0.5 - fyp;
            for (int j = 0; j < 2 * P.ry; ++j) {
                const long long yy = y0 + j;
                if (yy < 0 || yy >= P.Hs) continue;
                const double wy = tap_weight(P.kind, ((double)(j + 1 - P.ry) - ddy) * P.fy);
                if (wy == 0.0) continue;
                for (int i = 0; i < 2 * P.rx; ++i) {
                    const long long xx = x0 + i;
                    if (xx < 0 || xx >= P.Ws) continue;
                    const double w = (double)(float)(wy * tap_weight(P.kind, ((double)(i + 1 - P.rx) - ddx) * P.fx));
                    const long long s = yy * P.Ws + xx;
                    if (w == 0.0 || !__ldg(P.src_valid + s)) continue;
                    ws += w;
                    const float* sp = P.src + s;
#pragma unroll
                    for (int k = 0; k < K; ++k) acc[k] = fma(w, (double)__ldg(sp + k * P.src_plane_stride), acc[k]);
                }
            }
        }
        const bool covered = inside && ws >= 1e-6;
        bool fit = covered;
        float* dp = P.dst + o;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float v = covered ? (float)(acc[k] / ws) : __ldg(P.fill_out + k);
            dp[k * P.dst_plane_stride] = v;
            fit = fit && isfinite(v) && (k != P.gate_k || v > P.gate_gt);
        }
        if (P.dst_valid) P.dst_valid[o] = covered ? 1 : 0;
        if (P.fit_mask) P.fit_mask[o] = fit ? 1 : 0;
    }
}

template <int K>
void launch_warp_planes(dim3 grid, cudaStream_t stream, const PlaneParams& P) {
    warp_planes_kernel<K><<<grid, dim3(PL_COLS, PL_ROWS), 0, stream>>>(P);
}

// ---------------------------------------------------------------------------- host side
int fill_params(WarpParams& P, const hsr_warp_geo_t* geo, long long Hs, long long Ws, long long Hd, long long Wd,
                int kernel) {
    HSR_REQUIRE(geo, HSR_EINVAL, "null geo pointer");
    HSR_REQUIRE(kernel >= 0 && kernel <= 3, HSR_EINVAL,
                "kernel must be 0 (nearest), 1 (bilinear), 2 (cubic) or 3 (average), got %d", kernel);
    HSR_REQUIRE(geo->utm_zone >= 0 && geo->utm_zone <= 60, HSR_ERANGE, "utm_zone = %d outside [0, 60]", geo->utm_zone);
    const double* s = geo->src_gt;
    const double det = s[1] * s[5] - s[2] * s[4];
    HSR_REQUIRE(det != 0.0 && det == det, HSR_EINVAL, "source geotransform is singular");
    for (int i = 0; i < 6; ++i) P.dgt[i] = geo->dst_gt[i];
    P.sx0 = s[0];
    P.sy0 = s[3];
    P.inv[0] = s[5] / det;
    P.inv[1] = -s[2] / det;
    P.inv[2] = -s[4] / det;
    P.inv[3] = s[1] / det;
    P.utm = geo->utm_zone > 0 ? 1 : 0;
    if (P.utm) {    // WGS-84, k0 = 0.9996; Krueger series to n^6 (Karney 2011, eq. 36)
        const double a = 6378137.0, f = 1.0 / 298.257223563;
        const double n = f / (2.0 - f), n2 = n * n, n3 = n2 * n, n4 = n3 * n, n5 = n4 * n, n6 = n5 * n;
        const double A = a / (1.0 + n) * (1.0 + n2 / 4.0 + n4 / 64.0 + n6 / 256.0);
        P.k0A_inv = 1.0 / (0.9996 * A);
        P.e = sqrt(f * (2.0 - f));
        P.e2m = 1.0 - f * (2.0 - f);
        P.lon0_deg = -183.0 + 6.0 * geo->utm_zone;
        P.false_northing = geo->south ? 10000000.0 : 0.0;
        P.beta[0] = n / 2 - 2 * n2 / 3 + 37 * n3 / 96 - n4 / 360 - 81 * n5 / 512 + 96199 * n6 / 604800;
        P.beta[1] = n2 / 48 + n3 / 15 - 437 * n4 / 1440 + 46 * n5 / 105 - 1118711 * n6 / 3870720;
        P.beta[2] = 17 * n3 / 480 - 37 * n4 / 840 - 209 * n5 / 4480 + 5569 * n6 / 90720;
        P.beta[3] = 4397 * n4 / 161280 - 11 * n5 / 504 - 830251 * n6 / 7257600;
        P.beta[4] = 4583 * n5 / 161280 - 108847 * n6 / 3991680;
        P.beta[5] = 20648693 * n6 / 638668800;
    }
    P.Hs = Hs, P.Ws = Ws, P.Hd = Hd, P.Wd = Wd;
    P.kind = kernel;
    const int r0 = kernel == 2 ? 2 : 1;
    if (kernel == 0 || kernel == 3) {   // point kernels: no filter taps, the scales are not used
        P.fx = P.fy = 1.0;
        P.rx = P.ry = 1;
        return HSR_OK;
    }
    const double xs = geo->xscale > 0.0 ? geo->xscale : 1.0, ys = geo->yscale > 0.0 ? geo->yscale : 1.0;
    P.fx = xs < 1.0 ? xs : 1.0;
    P.fy = ys < 1.0 ? ys : 1.0;
    const double rxd = xs < 1.0 ? ceil(r0 / xs) : (double)r0, ryd = ys < 1.0 ? ceil(r0 / ys) : (double)r0;
    HSR_REQUIRE(rxd <= MAX_TAPS / 2 && ryd <= MAX_TAPS / 2, HSR_ERANGE,
                "scale (%g, %g) needs a filter radius beyond %d taps", xs, ys, MAX_TAPS / 2);
    P.rx = (int)rxd;
    P.ry = (int)ryd;
    return HSR_OK;
}

}  // namespace

// 3-D tensor map over the band-interleaved source cube: (bands, x, y) with byte strides (4, pixel stride, row stride);
// box {32 bands, bw pixels, bh rows}; out-of-range elements (outside the cube, bands beyond the last) read as zero.
// cuTensorMapEncodeTiled comes from the driver through the runtime's entry-point query: no link-time libcuda.
static int encode_src_map(CUtensorMap* map, const float* src, long long Hs, long long Ws, int bands, long long pix_stride,
                          int bw, int bh) {
    typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || !p ||
            qr != cudaDriverEntryPointSuccess)
            return HSR_EINVAL;
        fn = reinterpret_cast<encode_fn>(p);
    }
    const cuuint64_t dims[3] = {(cuuint64_t)bands, (cuuint64_t)Ws, (cuuint64_t)Hs};
    const cuuint64_t strides[2] = {(cuuint64_t)pix_stride * 4ull, (cuuint64_t)Ws * (cuuint64_t)pix_stride * 4ull};
    const cuuint32_t box[3] = {32u, (cuuint32_t)bw, (cuuint32_t)bh};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    if (strides[1] >= (1ull << 40)) return HSR_ERANGE;
    const CUresult rc = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(src), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return rc == CUDA_SUCCESS ? HSR_OK : HSR_EINVAL;
}

// warp_quad_kernel, if its two TMA buffers fit an SM next to the instantiation's static shared memory (`launched`;
// otherwise the caller takes the lane-per-pixel kernel).  TMA box = the tile's windows estimated from the scales (+ 1 of
// slack per axis for rotation / rounding; a tile that needs more reads its taps from global memory)
static int launch_warp_quad(const WarpParams& P, const hsr_warp_geo_t* geo, bool& launched, cudaStream_t stream) {
    launched = false;
    const double xs = geo->xscale > 0.0 ? geo->xscale : 1.0, ys = geo->yscale > 0.0 ? geo->yscale : 1.0;
    // source pixels per destination pixel, from the transformer itself at the grid's centre and corners (the
    // filter scales the caller passes need not describe the geometry)
    const long long Hd = P.Hd, Wd = P.Wd;
    double stepx = 1.0 / xs, stepy = 1.0 / ys;
    {
        const double cs[3] = {0.5, Wd * 0.5, Wd - 0.5}, rs[3] = {0.5, Hd * 0.5, Hd - 0.5};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double x0, y0, x1, y1, x2, y2;
                dst_to_src(P, cs[i], rs[j], x0, y0);
                dst_to_src(P, cs[i] + 1.0, rs[j], x1, y1);
                dst_to_src(P, cs[i], rs[j] + 1.0, x2, y2);
                // a tile's window origins span (QCOLS - 1) column steps and (QROWS - 1) row steps, in x AND in y
                const double sx = (fabs(x1 - x0) * (QCOLS - 1) + fabs(x2 - x0) * (QROWS - 1)) / (QCOLS - 1);
                const double sy = (fabs(y2 - y0) * (QROWS - 1) + fabs(y1 - y0) * (QCOLS - 1)) / (QROWS - 1);
                if (sx == sx && sx > stepx) stepx = sx;
                if (sy == sy && sy > stepy) stepy = sy;
            }
    }
    QuadGeo G{};
    // span of the window origins over the tile + the window + 1 of slack for rounding; kept tight: two CTAs of
    // 2 buffers each must fit an SM's 227 KB
    G.BW = (int)ceil((QCOLS - 1) * stepx) + 2 * P.rx + 1;
    G.BH = (int)ceil((QROWS - 1) * stepy) + 2 * P.ry + 1;
    const size_t qsmem_bytes = (size_t)2 * G.BW * G.BH * 128;
    CUtensorMap tmap;
    if (!(G.BW <= 256 && G.BH <= 256 && qsmem_bytes + 8192 <= (size_t)device_max_smem_optin() &&
          encode_src_map(&tmap, P.src, P.Hs, P.Ws, P.bands, P.src_pix_stride, G.BW, G.BH) == HSR_OK))
        return HSR_OK;
    const long long qtiles = ((Wd + QCOLS - 1) / QCOLS) * ((Hd + QROWS - 1) / QROWS);
    long long qblocks = (long long)device_sm_count() * 2;
    if (qblocks > qtiles) qblocks = qtiles;
// (the static shared memory of an instantiation — weight tables, class table — grows with the tap counts: the two
//  buffers must fit next to it, or the call takes the lane-per-pixel kernel; found by the fuzz soak, <8, 8>)
#define HSR_LAUNCH_QUAD(NX, NY)                                                                                           \
    do {                                                                                                                  \
        static int set__[HSR_MAX_DEVICES];                                                                                \
        static size_t static__ = 0;                                                                                       \
        if (static__ == 0) {                                                                                              \
            cudaFuncAttributes fa__;                                                                                      \
            HSR_CUDA(cudaFuncGetAttributes(&fa__, warp_quad_kernel<NX, NY, true>));                                       \
            static__ = fa__.sharedSizeBytes + 1;                                                                          \
        }                                                                                                                 \
        if (qsmem_bytes + static__ > (size_t)device_max_smem_optin()) return HSR_OK;                                      \
        HSR_CUDA(ensure_dynamic_smem(warp_quad_kernel<NX, NY, true>, (int)qsmem_bytes, set__));                           \
        warp_quad_kernel<NX, NY, true><<<(unsigned int)qblocks, 256, qsmem_bytes, stream>>>(tmap, P, G);                  \
    } while (0)
#define HSR_QUAD_Y(NX)                                  \
    do {                                                \
        if (P.ry == 1) HSR_LAUNCH_QUAD(NX, 2);          \
        else if (P.ry == 2) HSR_LAUNCH_QUAD(NX, 4);     \
        else if (P.ry == 3) HSR_LAUNCH_QUAD(NX, 6);     \
        else HSR_LAUNCH_QUAD(NX, 8);                    \
    } while (0)
    if (P.rx == 1) HSR_QUAD_Y(2);
    else if (P.rx == 2) HSR_QUAD_Y(4);
    else if (P.rx == 3) HSR_QUAD_Y(6);
    else HSR_QUAD_Y(8);
#undef HSR_QUAD_Y
#undef HSR_LAUNCH_QUAD
    launched = true;
    return HSR_OK;
}

// coordinates of every destination pixel (16 B each) + the fix-up list of the fast kernels (count word + entries)
static size_t warp_list_cap(long long Hd, long long Wd) {
    const long long n = Hd * Wd;
    return (size_t)(n < (1LL << 18) ? (n < 1024 ? 1024 : n) : (1LL << 18));
}
size_t warp_workspace(long long Hd, long long Wd) {
    return Hd > 0 && Wd > 0 ? (size_t)Hd * (size_t)Wd * 16 + 16 + warp_list_cap(Hd, Wd) * 8 : 0;
}

int warp_impl(const float* src, long long Hs, long long Ws, int bands, long long src_pix_stride, const hsr_warp_geo_t* geo,
              int kernel, int has_nodata, float nodata, float dst_nodata, long long Hd, long long Wd, float* dst,
              long long dst_pix_stride, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    HSR_REQUIRE(src && dst, HSR_EINVAL, "null src / dst pointer");
    HSR_REQUIRE(Hs > 0 && Ws > 0 && bands > 0 && Hd >= 0 && Wd >= 0, HSR_EINVAL, "bad shape");
    HSR_REQUIRE(Hs < 2147483000LL && Ws < 2147483000LL && Hs * Ws < (1LL << 40) && Hd * Wd < (1LL << 40), HSR_ERANGE,
                "grid too large (source sides are limited to 2^31 pixels, grids to 2^40)");
    HSR_REQUIRE(src_pix_stride >= bands && dst_pix_stride >= bands, HSR_EINVAL, "pixel stride < bands");
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 3) == 0, HSR_EALIGN,
                "src / dst not 4-byte aligned");
    WarpParams P{};
    int rc = fill_params(P, geo, Hs, Ws, Hd, Wd, kernel);
    if (rc != HSR_OK) return rc;
    if (Hd == 0 || Wd == 0) return HSR_OK;
    P.src = src;
    P.src_pix_stride = src_pix_stride;
    P.bands = bands;
    P.dst = dst;
    P.dst_pix_stride = dst_pix_stride;
    P.has_nodata = has_nodata ? 1 : 0;
    P.nodata = nodata;
    P.dst_nodata = dst_nodata;
    if (kernel == 0 || kernel == 3) {   // nearest / average: every pixel transforms its own centre or corners
        long long pb = (Hd * Wd + 255) / 256;
        const long long pcap = (long long)device_sm_count() * 16;
        warp_point_kernel<<<(unsigned int)(pb < pcap ? pb : pcap), 256, 0, stream>>>(P);
        HSR_CUDA(cudaGetLastError());
        return HSR_OK;
    }
    HSR_REQUIRE(workspace, HSR_EINVAL, "null workspace: kernels 1 (bilinear) and 2 (cubic) need hsr_warp_workspace_bytes(Hd, Wd)");
    HSR_REQUIRE(workspace_bytes >= warp_workspace(Hd, Wd), HSR_EINVAL, "workspace too small (%zu < %zu bytes)",
                workspace_bytes, warp_workspace(Hd, Wd));
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, HSR_EALIGN, "workspace not 16-byte aligned");
    // source coordinates of every destination pixel, once, instead of per tile and band group
    P.coords = static_cast<double*>(workspace);
    unsigned char* tail = static_cast<unsigned char*>(workspace) + (size_t)Hd * (size_t)Wd * 16;
    P.redo_count = reinterpret_cast<unsigned int*>(tail);
    P.redo_list = reinterpret_cast<unsigned long long*>(tail + 16);
    P.redo_cap = (unsigned int)warp_list_cap(Hd, Wd);
    long long cb = (Hd * Wd + 32 * WARPS - 1) / (32 * WARPS);
    const long long ccap = (long long)device_sm_count() * 8;
    warp_coords_kernel<<<(unsigned int)(cb < ccap ? cb : ccap), 32 * WARPS, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    HSR_CUDA(cudaMemsetAsync(P.redo_count, 0, 16, stream));
    const bool src_vec = (src_pix_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
    const bool dst_vec = (dst_pix_stride & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
    // the quad and lane kernels hold windows of up to 8 x 8 taps and index the source's pixels in 32 bits
    const bool narrow = P.rx <= 4 && P.ry <= 4 && Hs * Ws < 4294967295LL;
    bool quad = false;
    if (narrow && src_vec && dst_vec) {     // 2 x 2 block kernel, TMA-staged; declines when its buffers do not fit an SM
        rc = launch_warp_quad(P, geo, quad, stream);
        if (rc != HSR_OK) return rc;
    }
    if (!quad && narrow) {
        // lane-per-pixel kernel: register window of NT x NT taps, NT = 2 * max radius rounded up to 2, 4, 6, 8
        const int rmax = P.rx > P.ry ? P.rx : P.ry;
        const long long ltiles = ((Wd + LCOLS - 1) / LCOLS) * ((Hd + LROWS - 1) / LROWS);
        long long blocks = (long long)device_sm_count() * 3;
        if (blocks > ltiles) blocks = ltiles;
        const size_t smem = (size_t)LQ * LPITCH * sizeof(float4);
        const int sv = src_vec ? 1 : 0;
#define HSR_LAUNCH_LANE(NTV)                                                                                              \
    do {                                                                                                                  \
        if (dst_vec) {                                                                                                    \
            { static int set__[HSR_MAX_DEVICES]; HSR_CUDA(ensure_dynamic_smem(warp_lane_kernel<NTV, true>, (int)smem, set__)); } \
            warp_lane_kernel<NTV, true><<<(unsigned int)blocks, 256, smem, stream>>>(P, sv);                              \
        } else {                                                                                                          \
            { static int set__[HSR_MAX_DEVICES]; HSR_CUDA(ensure_dynamic_smem(warp_lane_kernel<NTV, false>, (int)smem, set__)); } \
            warp_lane_kernel<NTV, false><<<(unsigned int)blocks, 256, smem, stream>>>(P, sv);                             \
        }                                                                                                                 \
    } while (0)
        if (rmax <= 1) HSR_LAUNCH_LANE(2);
        else if (rmax == 2) HSR_LAUNCH_LANE(4);
        else if (rmax == 3) HSR_LAUNCH_LANE(6);
        else HSR_LAUNCH_LANE(8);
#undef HSR_LAUNCH_LANE
    } else if (!quad) {
        // the exact pass over every (pixel, quad): wider filters, sources of 2^32 pixels or more
        static int resident[HSR_MAX_DEVICES];
        long long blocks = (Hd * Wd * ((bands + 3) / 4) + 255) / 256;
        const long long cap = resident_blocks_cached(warp_exact_kernel, 256, resident);
        warp_exact_kernel<<<(unsigned int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(P, true);
    }
    HSR_CUDA(cudaGetLastError());
    // the fix-up: the entries the quad or lane kernel listed (the list is empty after the exact pass)
    warp_exact_kernel<<<(unsigned int)device_sm_count(), 256, 0, stream>>>(P, false);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int warp_coords_impl(const hsr_warp_geo_t* geo, long long Hd, long long Wd, double* coords, cudaStream_t stream) {
    HSR_REQUIRE(coords, HSR_EINVAL, "null coords pointer");
    HSR_REQUIRE(Hd >= 0 && Wd >= 0, HSR_EINVAL, "bad shape");
    WarpParams P{};
    int rc = fill_params(P, geo, 1, 1, Hd, Wd, 2);
    if (rc != HSR_OK) return rc;
    if (Hd == 0 || Wd == 0) return HSR_OK;
    P.coords = coords;
    long long blocks = (Hd * Wd + 32 * WARPS - 1) / (32 * WARPS);
    const long long cap = (long long)device_sm_count() * 8;
    if (blocks > cap) blocks = cap;
    warp_coords_kernel<<<(unsigned int)blocks, 32 * WARPS, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int warp_planes_impl(const float* src, long long Hs, long long Ws, int K, long long src_plane_stride,
                     const uint8_t* src_valid, const double* coords, const hsr_warp_geo_t* geo, int kernel,
                     const float* fill_out, int gate_k, float gate_gt, long long Hd, long long Wd, float* dst,
                     long long dst_plane_stride, uint8_t* dst_valid, uint8_t* fit_mask, cudaStream_t stream) {
    HSR_REQUIRE(src && dst && src_valid && fill_out, HSR_EINVAL, "null src / dst / src_valid / fill_out pointer");
    HSR_REQUIRE(coords, HSR_EINVAL, "null coords pointer: pass hsr_warp_coords_f64's output");
    HSR_REQUIRE(geo, HSR_EINVAL, "null geo pointer");
    HSR_REQUIRE(K >= 1 && K <= HSR_MAX_SRF_BANDS, HSR_EINVAL, "K = %d outside [1, %d]", K, HSR_MAX_SRF_BANDS);
    HSR_REQUIRE(kernel == 1 || kernel == 2, HSR_EINVAL, "kernel must be 1 (bilinear) or 2 (cubic), got %d", kernel);
    HSR_REQUIRE(Hs > 0 && Ws > 0 && Hd >= 0 && Wd >= 0, HSR_EINVAL, "bad shape");
    HSR_REQUIRE(Hs * Ws < (1LL << 40) && Hd * Wd < (1LL << 40), HSR_EINVAL, "grid too large (limit 2^40 pixels)");
    HSR_REQUIRE((K == 1 || src_plane_stride >= Hs * Ws) && (K == 1 || dst_plane_stride >= Hd * Wd) &&
                    src_plane_stride >= 0 && dst_plane_stride >= 0,
                HSR_EINVAL, "plane stride below the plane size");
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(coords) & 15) == 0, HSR_EALIGN, "coords not 16-byte aligned");
    HSR_REQUIRE(gate_k < K, HSR_EINVAL, "gate_k = %d >= K = %d", gate_k, K);
    PlaneParams P{};
    const int r0 = kernel == 2 ? 2 : 1;
    const double xs = geo->xscale > 0.0 ? geo->xscale : 1.0, ys = geo->yscale > 0.0 ? geo->yscale : 1.0;
    const double rxd = xs < 1.0 ? ceil(r0 / xs) : (double)r0, ryd = ys < 1.0 ? ceil(r0 / ys) : (double)r0;
    HSR_REQUIRE(rxd <= MAX_TAPS / 2 && ryd <= MAX_TAPS / 2, HSR_EINVAL,
                "scale (%g, %g) needs a filter radius beyond %d taps", xs, ys, MAX_TAPS / 2);
    if (Hd == 0 || Wd == 0) return HSR_OK;
    P.src = src;
    P.src_valid = src_valid;
    P.Hs = Hs, P.Ws = Ws, P.src_plane_stride = src_plane_stride;
    P.coords = coords;
    P.Hd = Hd, P.Wd = Wd;
    P.kind = kernel;
    P.rx = (int)rxd, P.ry = (int)ryd;
    P.fx = xs < 1.0 ? xs : 1.0;
    P.fy = ys < 1.0 ? ys : 1.0;
    P.fill_out = fill_out;
    P.gate_k = gate_k;
    P.gate_gt = gate_gt;
    P.dst = dst;
    P.dst_plane_stride = dst_plane_stride;
    P.dst_valid = dst_valid;
    P.fit_mask = fit_mask;
    const long long tiles_x = (Wd + PL_COLS - 1) / PL_COLS, tiles_y = (Hd + PL_ROWS - 1) / PL_ROWS;
    HSR_REQUIRE(tiles_x < 2147483647LL, HSR_EINVAL, "destination too wide");
    const dim3 grid((unsigned int)tiles_x, (unsigned int)(tiles_y < 65535 ? tiles_y : 65535));
    typedef void (*launch_fn)(dim3, cudaStream_t, const PlaneParams&);
    static const launch_fn launch[HSR_MAX_SRF_BANDS] = {
        launch_warp_planes<1>,  launch_warp_planes<2>,  launch_warp_planes<3>,  launch_warp_planes<4>,
        launch_warp_planes<5>,  launch_warp_planes<6>,  launch_warp_planes<7>,  launch_warp_planes<8>,
        launch_warp_planes<9>,  launch_warp_planes<10>, launch_warp_planes<11>, launch_warp_planes<12>,
        launch_warp_planes<13>, launch_warp_planes<14>, launch_warp_planes<15>, launch_warp_planes<16>};
    launch[K - 1](grid, stream, P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

}  // namespace hsr
