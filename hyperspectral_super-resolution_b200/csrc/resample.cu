// resample.cu — grid resampling, the ALIGNED INTEGER-RATIO case of SURVEY section 8f row 4: bringing the Sentinel-2
// 10 m stack onto the EMIT 60 m grid with "average" resampling (the notebook's downsample_s2_to_grid,
// Pairs_EMIT_S2_demo-2.ipynb cell 73, called at s2_emit/poly_regression.py:110-116 with src_scale = 1/255).
// nc_to_envi snaps the EMIT grid to the Sentinel-2 origin with an integer pixel ratio (emit_proj.py:794-797), so
// every 60 m pixel covers exactly factor x factor 10 m pixels and GDAL's average is their plain mean (nodata
// pixels excluded; no valid pixel -> the destination keeps its initial 0).  Parity with GDAL itself is UNPINNED
// (no GDAL / rasterio in the build image); general warps (other CRS, rotation, cubic, bilinear) are out of scope.
// One thread per output pixel; a warp covers 32 consecutive outputs, i.e. a contiguous span of every source row.
#include "hsr_common.cuh"

namespace hsr {

namespace {

template <typename T>
__global__ void __launch_bounds__(256) block_average_kernel(const T* __restrict__ src, long long src_plane_stride,
                                                            long long Ws, int factor, long long Hd, long long Wd,
                                                            int has_nodata, double nodata, float scale, int has_scale,
                                                            float* __restrict__ dst, long long dst_plane_stride) {
    const long long c = blockIdx.y;
    const T* sp = src + c * src_plane_stride;
    float* dp = dst + c * dst_plane_stride;
    const long long n = Hd * Wd;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < n; o += (long long)gridDim.x * blockDim.x) {
        const long long y = o / Wd, x = o - y * Wd;
        const T* blk = sp + (y * factor) * Ws + x * factor;
        double sum = 0.0;
        int cnt = 0;
        for (int r = 0; r < factor; ++r) {
            const T* row = blk + (long long)r * Ws;
            for (int q = 0; q < factor; ++q) {
                const double v = (double)row[q];
                const bool use = !(has_nodata && v == nodata) && v == v;
                sum += use ? v : 0.0;
                cnt += use ? 1 : 0;
            }
        }
        float out = cnt ? (float)(sum / (double)cnt) : 0.f;
        if (has_scale) out = __fmul_rn(out, scale);   // `out *= float(src_scale)` on the float32 result
        dp[o] = out;
    }
}

}  // namespace

int block_average_impl(const void* src, int src_dtype, int C, long long Hs, long long Ws, long long src_plane_stride,
                       int factor, int has_nodata, double nodata, int has_scale, float scale, float* dst,
                       long long dst_plane_stride, cudaStream_t stream) {
    HSR_REQUIRE(src && dst, HSR_EINVAL, "null src / dst pointer");
    HSR_REQUIRE(C >= 1 && C <= 65535 && Hs >= 0 && Ws >= 0 && factor >= 1, HSR_EINVAL, "bad shape or factor");
    HSR_REQUIRE(src_dtype >= 0 && src_dtype <= 2, HSR_EINVAL, "src_dtype must be 0 (u8), 1 (u16) or 2 (f32)");
    const long long Hd = Hs / factor, Wd = Ws / factor;
    HSR_REQUIRE(src_plane_stride >= Hs * Ws && dst_plane_stride >= Hd * Wd, HSR_EINVAL, "plane stride too small");
    if (Hd == 0 || Wd == 0) return HSR_OK;
    long long blocks = (Hd * Wd + 255) / 256;
    long long cap = (long long)device_sm_count() * 8 / C;
    if (cap < 1) cap = 1;
    dim3 grid((unsigned int)(blocks < cap ? blocks : cap), (unsigned int)C);
    if (src_dtype == 0)
        block_average_kernel<uint8_t><<<grid, 256, 0, stream>>>(static_cast<const uint8_t*>(src), src_plane_stride, Ws, factor,
                                                               Hd, Wd, has_nodata, nodata, scale, has_scale, dst,
                                                               dst_plane_stride);
    else if (src_dtype == 1)
        block_average_kernel<uint16_t><<<grid, 256, 0, stream>>>(static_cast<const uint16_t*>(src), src_plane_stride, Ws,
                                                                factor, Hd, Wd, has_nodata, nodata, scale, has_scale, dst,
                                                                dst_plane_stride);
    else
        block_average_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(src), src_plane_stride, Ws, factor, Hd,
                                                             Wd, has_nodata, nodata, scale, has_scale, dst, dst_plane_stride);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

}  // namespace hsr

namespace hsr {

namespace {

// Bilinear resampling onto a `factor`-times FINER aligned grid (the notebook's reproject_stack_to_grid with
// Resampling.bilinear, cell 73; s2_emit/poly_regression.py:150-156): the destination pixel centre
// ((x + 0.5) / factor - 0.5 in source pixel coordinates) is interpolated from its 2 x 2 source neighbours; neighbours
// outside the source, equal to nodata or NaN are skipped and the weights renormalised (GDAL's 4-sample bilinear
// kernel), none usable -> 0.  fp64 weights, fp32 result (bilinear_up_tap / bilinear_up_value of hsr_common.cuh).
__global__ void __launch_bounds__(256) bilinear_up_kernel(const float* __restrict__ src, long long src_plane_stride,
                                                          long long Hs, long long Ws, int factor, int has_nodata,
                                                          float nodata, float* __restrict__ dst,
                                                          long long dst_plane_stride) {
    const long long c = blockIdx.y;
    const float* sp = src + c * src_plane_stride;
    float* dp = dst + c * dst_plane_stride;
    const long long Hd = Hs * factor, Wd = Ws * factor, n = Hd * Wd;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < n; o += (long long)gridDim.x * blockDim.x) {
        const long long y = o / Wd, x = o - y * Wd;
        dp[o] = bilinear_up_value(sp, Hs, Ws, bilinear_up_tap(y, x, factor), has_nodata, nodata);
    }
}

}  // namespace

int bilinear_upsample_impl(const float* src, int C, long long Hs, long long Ws, long long src_plane_stride, int factor,
                           int has_nodata, float nodata, float* dst, long long dst_plane_stride, cudaStream_t stream) {
    HSR_REQUIRE(src && dst, HSR_EINVAL, "null src / dst pointer");
    HSR_REQUIRE(C >= 1 && C <= 65535 && Hs >= 0 && Ws >= 0 && factor >= 1, HSR_EINVAL, "bad shape or factor");
    HSR_REQUIRE(src_plane_stride >= Hs * Ws && dst_plane_stride >= Hs * Ws * factor * factor, HSR_EINVAL,
                "plane stride too small");
    if (Hs == 0 || Ws == 0) return HSR_OK;
    long long blocks = (Hs * Ws * factor * factor + 255) / 256;
    long long cap = (long long)device_sm_count() * 8 / C;
    if (cap < 1) cap = 1;
    dim3 grid((unsigned int)(blocks < cap ? blocks : cap), (unsigned int)C);
    bilinear_up_kernel<<<grid, 256, 0, stream>>>(src, src_plane_stride, Hs, Ws, factor, has_nodata, nodata, dst,
                                                 dst_plane_stride);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

namespace {

// mask10 of s2_emit/poly_regression.py:159: mask[i] = all_k isfinite(bilinear x factor of plane k at fine pixel i),
// computed from the source planes without writing the fine planes.  One thread per 4 fine pixels of the flat index.
__global__ void __launch_bounds__(256) bilinear_fine_mask_kernel(const float* __restrict__ src, int K,
                                                                 long long src_plane_stride, long long Hs,
                                                                 long long Ws, int factor, uint8_t* __restrict__ mask,
                                                                 int vecm) {
    const long long Wd = Ws * factor, n = Hs * factor * Wd, n4 = (n + 3) >> 2;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n4; q += (long long)gridDim.x * blockDim.x) {
        const long long i = q << 2;
        long long y = i / Wd, x = i - y * Wd;
        BilinearTap t[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            t[j] = bilinear_up_tap(y, x, factor);
            next_pixel(y, x, Wd);
        }
        unsigned int m = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) m |= (i + j < n ? 1u : 0u) << j;
        for (int k = 0; k < K; ++k) {
            const float* sp = src + (long long)k * src_plane_stride;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (((m >> j) & 1u) && !finite_f32(bilinear_up_value(sp, Hs, Ws, t[j], 0, 0.f))) m &= ~(1u << j);
        }
        if (vecm && i + 4 <= n) {
            *reinterpret_cast<uchar4*>(mask + i) = make_uchar4(m & 1u, (m >> 1) & 1u, (m >> 2) & 1u, (m >> 3) & 1u);
        } else {
            for (int j = 0; j < 4; ++j)
                if (i + j < n) mask[i + j] = (m >> j) & 1u;
        }
    }
}

}  // namespace

int bilinear_fine_mask_impl(const float* src, int K, long long Hs, long long Ws, long long src_plane_stride, int factor,
                            uint8_t* mask, cudaStream_t stream) {
    HSR_REQUIRE(src && mask, HSR_EINVAL, "null src / mask pointer");
    HSR_REQUIRE(K >= 1 && K <= HSR_MAX_SRF_BANDS && Hs >= 0 && Ws >= 0 && factor >= 1, HSR_EINVAL,
                "bad K = %d (1..%d), shape or factor", K, HSR_MAX_SRF_BANDS);
    HSR_REQUIRE(src_plane_stride >= Hs * Ws, HSR_EINVAL, "plane stride too small");
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(src) & 3) == 0, HSR_EALIGN, "src not 4-byte aligned");
    if (Hs == 0 || Ws == 0) return HSR_OK;
    const long long n4 = (Hs * Ws * factor * factor + 3) / 4;
    long long blocks = (n4 + 255) / 256;
    const long long cap = (long long)device_sm_count() * 8;
    const int vecm = (reinterpret_cast<uintptr_t>(mask) & 3) == 0 ? 1 : 0;
    bilinear_fine_mask_kernel<<<(unsigned int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(
        src, K, K > 1 ? src_plane_stride : Hs * Ws, Hs, Ws, factor, mask, vecm);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

}  // namespace hsr
