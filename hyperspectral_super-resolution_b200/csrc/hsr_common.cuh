// hsr_common.cuh — sm_100a building blocks shared by the hot-path kernels:
// mbarrier + 1-D bulk-copy (TMA, SASS UBLKCP) wrappers, warp reductions, error plumbing.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/hsr_b200.h"

namespace hsr {

// ---------------------------------------------------------------- error plumbing (thread-local)
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define HSR_REQUIRE(cond, code, ...)      \
    do {                                  \
        if (!(cond)) {                    \
            ::hsr::set_error(__VA_ARGS__); \
            return (code);                \
        }                                 \
    } while (0)

#define HSR_CUDA(call)                                          \
    do {                                                        \
        cudaError_t e__ = (call);                               \
        if (e__ != cudaSuccess) return ::hsr::cuda_fail(e__, #call); \
    } while (0)

int device_sm_count();          // cached per device
int device_max_smem_optin();    // cached per device
int current_device_slot();      // cudaGetDevice(), clamped to [0, HSR_MAX_DEVICES)

constexpr int HSR_MAX_DEVICES = 64;

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel instantiation, device) instead of on every
// launch: `cache` is a zero-initialised static int[HSR_MAX_DEVICES] owned by the caller's instantiation and
// remembers the largest size set so far.  Racing threads may both set the attribute — harmless.
template <typename Kern>
inline cudaError_t ensure_dynamic_smem(Kern kern, int bytes, int* cache) {
    const int d = current_device_slot();
    if (__atomic_load_n(&cache[d], __ATOMIC_RELAXED) >= bytes) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) __atomic_store_n(&cache[d], bytes, __ATOMIC_RELAXED);
    return e;
}

// cudaOccupancyMaxActiveBlocksPerMultiprocessor x SM count, cached the same way (0 dynamic shared memory).
template <typename Kern>
inline int resident_blocks_cached(Kern kern, int threads, int* cache) {
    const int d = current_device_slot();
    int r = __atomic_load_n(&cache[d], __ATOMIC_RELAXED);
    if (r > 0) return r;
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, threads, 0) != cudaSuccess || nb < 1) nb = 1;
    r = nb * device_sm_count();
    __atomic_store_n(&cache[d], r, __ATOMIC_RELAXED);
    return r;
}

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t tx_bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(tx_bytes)
                 : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
#ifdef HSR_MBAR_HINT_NS
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"   // may stay suspended up to the hint (ns)
#else
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#endif
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
#ifdef HSR_MBAR_HINT_NS
        : "r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)HSR_MBAR_HINT_NS)
#else
        : "r"(smem_u32(bar)), "r"(parity)
#endif
        : "memory");
    return done != 0;
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// 1-D bulk asynchronous copy global -> shared (TMA unit; completes on an mbarrier).
// dst, src 16-byte aligned; bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// L2 eviction-priority policies for data that is read exactly once (keeps re-used planes resident in the 126 MB L2).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar,
                                              uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ bool finite_f32(float v) {
    return (__float_as_uint(v) & 0x7f800000u) != 0x7f800000u;
}

// np.isclose(x, y, atol) on a float32 array against a Python float (finite y): float32 arithmetic, tol = f32(atol + rtol |y|)
__device__ __forceinline__ bool close32(float x, float y, float tol) {
    return fabsf(__fsub_rn(x, y)) <= tol || x == y;
}

// ---------------------------------------------------------------- bilinear x factor onto an aligned finer grid
// The 2 x 2 fp64 interpolation of hsr_bilinear_upsample_f32 (s2_emit/poly_regression.py:150-156), split so that a
// kernel mapping several planes at one fine pixel forms the pixel's taps once.  The destination pixel centre
// ((x + 0.5) / factor - 0.5 in source pixel coordinates) is interpolated from its 2 x 2 source neighbours; neighbours
// outside the source, equal to nodata or NaN are skipped and the weights renormalised, none usable -> 0.  Every kernel
// that resamples this way goes through these two helpers, so their fine values carry the same bits.
struct BilinearTap {
    long long y0, x0;
    double wy1, wx1;
};

__device__ __forceinline__ BilinearTap bilinear_up_tap(long long y, long long x, int factor) {
    const double sy = ((double)y + 0.5) / factor - 0.5, sx = ((double)x + 0.5) / factor - 0.5;
    const double fy = floor(sy), fx = floor(sx);
    return {(long long)fy, (long long)fx, sy - fy, sx - fx};
}

__device__ __forceinline__ float bilinear_up_value(const float* __restrict__ sp, long long Hs, long long Ws,
                                                   const BilinearTap& t, int has_nodata, float nodata) {
    double acc = 0.0, wsum = 0.0;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
        const long long yy = t.y0 + dy;
        const double wy = dy ? t.wy1 : 1.0 - t.wy1;
        if (yy < 0 || yy >= Hs) continue;
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const long long xx = t.x0 + dx;
            const double w = wy * (dx ? t.wx1 : 1.0 - t.wx1);
            if (xx < 0 || xx >= Ws || w == 0.0) continue;
            const float v = __ldg(sp + yy * Ws + xx);
            if ((has_nodata && v == nodata) || v != v) continue;
            acc += w * (double)v;
            wsum += w;
        }
    }
    return wsum > 0.0 ? (float)(acc / wsum) : 0.f;
}

// fine (y, x) of flat index i of a plane Wd wide, then of i + 1 (no division)
__device__ __forceinline__ void next_pixel(long long& y, long long& x, long long Wd) {
    if (++x == Wd) x = 0, ++y;
}

// tiles_helpers/utils.py:357-371: valid = isfinite(v) & (v != nodata); clip(int32(rint(v * scale)), 0, hi), nd otherwise.
// rint by the 1.5 * 2^23 trick (round-to-nearest-even of the clamped product; exact for 0 <= t <= 65534); a product
// beyond int32 converts to INT_MIN on x86 (numpy's astype) and is therefore clipped to 0.
__device__ __forceinline__ unsigned short quant_u16(float v, int has_nodata, float nodata, float scale, float hi,
                                                    unsigned short nd) {
    const bool valid = finite_f32(v) && !(has_nodata && v == nodata);
    const float r = __fmul_rn(v, scale);
    const float t = fminf(fmaxf(r, 0.f), hi);
    unsigned int q = __float_as_uint(__fadd_rn(t, 12582912.f)) & 0xffffu;
    if (!(fabsf(r) < 2147483648.f)) q = 0u;
    return valid ? (unsigned short)q : nd;
}

}  // namespace hsr
