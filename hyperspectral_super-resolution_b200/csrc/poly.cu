// poly.cu — kernel 3 of the hot path: per-series polynomial regression
//   moments (block-then-grid fp64 reduction of the normal equations X^T X / X^T y)
//   -> warp-level solve of the column-scaled system -> fused Horner apply + mask + clip.
// Arithmetic follows np.polyfit as called at s2_emit/poly_regression.py:58-60 and
// apply_poly_rgb at s2_emit/poly_regression.py:65-84.
#include <stdlib.h>
#include <string.h>

#include "hsr_common.cuh"

namespace hsr {

namespace {

constexpr int MAXDEG = HSR_MAX_POLY_DEG;
constexpr int MOM_THREADS = 256;

__host__ __device__ inline int n_moments(int deg) { return 3 * deg + 2; }

// One sample into the 3*DEG+2 sums: S_j = sum x^j (j = 0..2*DEG), T_j = sum x^j y (j = 0..DEG).
// Only the powers up to DEG are formed (DEG-1 multiplies); every higher S_j is a single fused
// multiply-add of two of them (x^a * x^b, a + b = j, rounded once), so a degree-2 sample costs 8
// fp64 operations.  x is fp32, so x and x^2 are exact in fp64.
template <int DEG>
__device__ __forceinline__ void accumulate(double (&acc)[3 * DEG + 2], float xf, float yf, bool use) {
    if (!use) return;
    const double x = (double)xf, y = (double)yf;
    double pw[DEG + 1];
    pw[0] = 1.0;
#pragma unroll
    for (int j = 1; j <= DEG; ++j) pw[j] = pw[j - 1] * x;
    acc[0] += 1.0;
    acc[1] += x;
#pragma unroll
    for (int j = 2; j <= 2 * DEG; ++j) acc[j] = fma(pw[j / 2], pw[j - j / 2], acc[j]);
    acc[2 * DEG + 1] += y;
#pragma unroll
    for (int j = 1; j <= DEG; ++j) acc[2 * DEG + 1 + j] = fma(pw[j], y, acc[2 * DEG + 1 + j]);
}

// s2_emit/color.py:33: np.clip((img - lo) / (hi - lo + 1e-12), 0, 1) in float64, stored as float32.
// The fused fit / apply kernels evaluate the quotient as a * rcp with one Newton correction (q + fma(-q, den, a) * rcp:
// within 1 ulp of the correctly rounded fp64 quotient) instead of an fp64 division per sample (~40 instructions: it
// tripled the moment kernel's time).  After the cast to float32 that differs from numpy's value for about one sample
// in 2^29 and by one float32 ulp — invisible in the fp64 moments and far inside the 1e-4 bars; the stand-alone
// hsr_stretch_f32 / hsr_stretch_f64 keep the true division and stay bit-exact.
__device__ __forceinline__ float stretch1(float v, double lo, double den, double rcp) {
    const double a = (double)v - lo;
    double r = a * rcp;
    r = fma(fma(-r, den, a), rcp, r);
    r = r < 0.0 ? 0.0 : (r > 1.0 ? 1.0 : r);  // NaN survives both comparisons, as np.clip
    return (float)r;
}

__device__ __forceinline__ float4 stretch4(float4 v, double lo, double den, double rcp) {
    return make_float4(stretch1(v.x, lo, den, rcp), stretch1(v.y, lo, den, rcp), stretch1(v.z, lo, den, rcp),
                       stretch1(v.w, lo, den, rcp));
}

// Moments of S = K * G series (series s = k * G + g at x + k * xks + g * xgs + i * xns).
// grid = (blocks per series, S).  Each thread keeps 3*DEG+2 fp64 accumulators (two 16-byte loads of x
// and of y in flight per thread on the vector path), the block reduces them by warp shuffles + shared
// memory and writes ONE partial row; moments_finalize_kernel then sums the rows of a series in a fixed
// order (bit-reproducible).  A sample is used iff its mask byte is set and x, y are finite
// (poly_regression.py:35-36).  STRETCH: x and y first go through the shared percentile stretch of
// s2_emit/color.py:25-34 (poly_regression.py:126-127), which is never materialised.
struct MomParams {
    const float* x;
    long long xks, xgs, xns;
    const float* y;
    long long yks, ygs, yns;
    const uint8_t* mask;  // nullable; series s uses row (s / mdiv) % mmod of n bytes
    long long mdiv, mmod;
    const double* xst;  // nullable [S][2] (lo, hi)
    const double* yst;
    long long n;
    int G;
    int reverse;  // hsr_fit_moments_f64 walks the samples from the end: the planes were just written front to back
                  // by the producer kernel, so their tail is what is still in L2 (a forward scan of 135 MB through a
                  // 126 MB LRU cache would miss everywhere).  hsr_poly_moments_f64 walks forward.
    double* partial;
};

template <int DEG, bool STRETCH>
__global__ void __launch_bounds__(MOM_THREADS) poly_moments_kernel(const MomParams P) {
    constexpr int M = 3 * DEG + 2;
    const long long s = blockIdx.y;
    const long long k = s / P.G, g = s - k * P.G;
    const long long n = P.n;
    const float* xk = P.x + k * P.xks + g * P.xgs;
    const float* yk = P.y + k * P.yks + g * P.ygs;
    const uint8_t* mk = P.mask ? P.mask + ((s / P.mdiv) % P.mmod) * n : nullptr;
    double xlo = 0.0, xden = 1.0, ylo = 0.0, yden = 1.0, xrcp = 1.0, yrcp = 1.0;
    bool sx = false, sy = false;
    if (STRETCH) {
        if (P.xst) sx = true, xlo = P.xst[2 * s], xden = P.xst[2 * s + 1] - xlo + 1e-12, xrcp = 1.0 / xden;
        if (P.yst) sy = true, ylo = P.yst[2 * s], yden = P.yst[2 * s + 1] - ylo + 1e-12, yrcp = 1.0 / yden;
    }

    double acc[M];
#pragma unroll
    for (int j = 0; j < M; ++j) acc[j] = 0.0;

    auto take = [&](float xv, float yv, bool m) {
        if (STRETCH) {
            if (sx) xv = stretch1(xv, xlo, xden, xrcp);
            if (sy) yv = stretch1(yv, ylo, yden, yrcp);
        }
        accumulate<DEG>(acc, xv, yv, m && finite_f32(xv) && finite_f32(yv));
    };
    auto take4 = [&](const float4 xv, const float4 yv, const uchar4 mv) {
        take(xv.x, yv.x, mv.x != 0);
        take(xv.y, yv.y, mv.y != 0);
        take(xv.z, yv.z, mv.z != 0);
        take(xv.w, yv.w, mv.w != 0);
    };

    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const bool vec = P.xns == 1 && P.yns == 1 &&
                     ((reinterpret_cast<uintptr_t>(xk) | reinterpret_cast<uintptr_t>(yk)) & 15) == 0 &&
                     (mk == nullptr || (reinterpret_cast<uintptr_t>(mk) & 3) == 0);
    long long done = 0;
    if (vec) {
        const long long n4 = n >> 2;
        const float4* x4 = reinterpret_cast<const float4*>(xk);
        const float4* y4 = reinterpret_cast<const float4*>(yk);
        const uchar4* m4 = reinterpret_cast<const uchar4*>(mk);
        const long long last = n4 - 1;
        long long i = tid;
        for (; i + nthreads < n4; i += 2 * nthreads) {
            const long long ia = P.reverse ? last - i : i, ib = P.reverse ? last - i - nthreads : i + nthreads;
            const float4 xa = __ldg(x4 + ia), xb = __ldg(x4 + ib);
            const float4 ya = __ldcs(y4 + ia), yb = __ldcs(y4 + ib);
            uchar4 ma = make_uchar4(1, 1, 1, 1), mb = ma;
            if (mk) ma = __ldg(m4 + ia), mb = __ldg(m4 + ib);
            take4(xa, ya, ma);
            take4(xb, yb, mb);
        }
        for (; i < n4; i += nthreads) {
            const long long ia = P.reverse ? last - i : i;
            uchar4 ma = make_uchar4(1, 1, 1, 1);
            if (mk) ma = __ldg(m4 + ia);
            take4(__ldg(x4 + ia), __ldcs(y4 + ia), ma);
        }
        done = n4 << 2;
    }
    for (long long i = done + tid; i < n; i += nthreads)
        take(__ldg(xk + i * P.xns), __ldg(yk + i * P.yns), mk == nullptr || mk[i] != 0);

    __shared__ double red[MOM_THREADS / 32][M];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < M; ++j) {
        const double t = warp_sum(acc[j]);
        if (lane == 0) red[warp][j] = t;
    }
    __syncthreads();
    if (threadIdx.x < M) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < MOM_THREADS / 32; ++w) t += red[w][threadIdx.x];
        P.partial[(s * gridDim.x + blockIdx.x) * M + threadIdx.x] = t;
    }
}

// ------------------------------------------------------------------------------------------------
// Cross-GPU exchange of the moments over NVLink peer memory (replaces the NCCL all-reduce of the fit).
// Every rank owns one PeerBlock in device memory, mapped into every other process by CUDA IPC.  The finalize
// kernel of rank r stores its S*M sums into slot r of EVERY rank's block (remote stores over NVLink / NVSwitch),
// fences, and the last of its blocks raises flag r there to the current epoch.  The solve/apply kernel of each rank
// polls its OWN block until all flags carry the epoch, adds the slots in rank order (bit-identical on every
// rank and run to run) and solves.  Two slot sets alternate by epoch parity: a rank can only be one epoch ahead
// of the slowest consumer, because its next finalize follows its own solve/apply, which waited for everyone.
constexpr int PEER_MAXR = HSR_PEER_MAX_RANKS;
constexpr int PEER_MAXD = HSR_PEER_MAX_DOUBLES;

struct PeerBlock {
    unsigned long long flags[2][PEER_MAXR];
    unsigned int ticket;
    unsigned int error;        // sticky status word: HSR_PEER_TIMEOUT once a solve/apply gave up waiting for a peer
    unsigned long long epoch;  // exchanges this rank has published (device-side epoch counter)
    double slots[2][PEER_MAXR][PEER_MAXD];
};

struct Exchange {       // device-side view (by value in the kernel parameters)
    PeerBlock* const* peers;  // device array [nranks]
    PeerBlock* mine;
    int nranks, rank;
    unsigned long long epoch;  // 0: take the epoch from the block's own counter (lets the step be replayed from a
                               // CUDA graph: nothing in the kernel parameters changes from exchange to exchange)
    unsigned long long timeout_ns;  // how long a solve/apply block waits for the peers' flags before it gives up
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Wait until flag >= epoch.  Bounded: a peer that died, raised before its finalize or runs fewer exchanges must not
// hang this GPU.  After timeout_ns (or as soon as another block of this kernel has already given up) the wait ends
// with `false` and the block's status word carries HSR_PEER_TIMEOUT for the host (hsr_peer_status).
__device__ __forceinline__ bool wait_flag(const unsigned long long* flag, unsigned long long epoch, PeerBlock* mine,
                                          unsigned long long timeout_ns) {
    if (ld_acquire_sys(flag) >= epoch) return true;
    const unsigned long long t0 = globaltimer_ns();
    for (unsigned int spin = 1;; ++spin) {
        if (ld_acquire_sys(flag) >= epoch) return true;
        if ((spin & 63u) == 0u) {
            if (*(volatile unsigned int*)&mine->error != 0u) return false;
            if (globaltimer_ns() - t0 > timeout_ns) {
                atomicOr(&mine->error, (unsigned int)HSR_PEER_TIMEOUT);
                __threadfence_system();
                return false;
            }
        }
    }
}

// Sum the partial rows of one series in a fixed order: 8 warps take rows w, w + 8, ... (lane = moment
// index), then the 8 slice sums are added in order.  One block per series.  With an exchange, the sums also go
// to every rank's peer block (see above).
__global__ void __launch_bounds__(256) moments_finalize_kernel(const double* __restrict__ partial, int rows, int M,
                                                               double* __restrict__ moments, const Exchange ex) {
    __shared__ double red[8][32];
    const long long s = blockIdx.x;
    const int j = threadIdx.x & 31, w = threadIdx.x >> 5;
    double a0 = 0.0, a1 = 0.0;
    if (j < M) {
        const double* p = partial + s * rows * (long long)M + j;
        int r = w;
        for (; r + 8 < rows; r += 16) {
            a0 += p[(long long)r * M];
            a1 += p[(long long)(r + 8) * M];
        }
        if (r < rows) a0 += p[(long long)r * M];
    }
    red[w][j] = a0 + a1;
    __syncthreads();
    if (w == 0 && j < M) {
        double t = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) t += red[q][j];
        moments[s * M + j] = t;
    }
    if (ex.nranks > 1) {
        // the epoch being published: the host's, or one more than this rank has published so far (every block reads
        // the counter before it takes its ticket; only the last block, after all tickets, advances it)
        const unsigned long long epoch = ex.epoch ? ex.epoch : *(volatile unsigned long long*)&ex.mine->epoch + 1ull;
        const int par = (int)(epoch & 1ull);
        if (w == 0 && j < M) {
            const double t = moments[s * M + j];
            for (int q = 0; q < ex.nranks; ++q) ex.peers[q]->slots[par][ex.rank][s * M + j] = t;
        }
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            if (atomicAdd(&ex.mine->ticket, 1u) == gridDim.x - 1) {  // every series of this rank is on its way
                ex.mine->ticket = 0u;
                ex.mine->epoch = epoch;
                __threadfence_system();
                for (int q = 0; q < ex.nranks; ++q) st_release_sys(&ex.peers[q]->flags[par][ex.rank], epoch);
            }
        }
    }
}

// Fixed-order sum of the moment matrices of this rank's units (granules of a shard): out[j] = sum_u per_unit[u][j],
// u ascending — bit-reproducible — and, with an exchange, the publication of the sums to every rank's peer block
// (same protocol as moments_finalize_kernel; one thread per moment).  This is the "local sum" of a global fit over
// many granules per rank (BASELINE configs[3]); the solve/apply of the FIRST granule then consumes the exchange.
__global__ void __launch_bounds__(256) moments_sum_kernel(const double* __restrict__ per_unit, int units,
                                                          long long count, double* __restrict__ out,
                                                          const Exchange ex) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    double t = 0.0;
    if (j < count)
        for (int u = 0; u < units; ++u) t += per_unit[(long long)u * count + j];
    if (j < count) out[j] = t;
    if (ex.nranks > 1) {
        const unsigned long long epoch = ex.epoch ? ex.epoch : *(volatile unsigned long long*)&ex.mine->epoch + 1ull;
        const int par = (int)(epoch & 1ull);
        if (j < count)
            for (int q = 0; q < ex.nranks; ++q) ex.peers[q]->slots[par][ex.rank][j] = t;
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            if (atomicAdd(&ex.mine->ticket, 1u) == gridDim.x - 1) {
                ex.mine->ticket = 0u;
                ex.mine->epoch = epoch;
                __threadfence_system();
                for (int q = 0; q < ex.nranks; ++q) st_release_sys(&ex.peers[q]->flags[par][ex.rank], epoch);
            }
        }
    }
}

// One warp solves one series, entirely in registers.  Normal equations G c = r with G_ij = S_{i+j},
// r_i = T_i, scaled by s_j = sqrt(S_{2j}) (the column norms np.polyfit divides its Vandermonde by),
// solved by Gauss-Jordan elimination with partial pivoting: lane j < N owns column j of the augmented
// matrix, lane N the right-hand side (lanes beyond N shadow lane N); pivots and multipliers travel
// by warp shuffles, so there is no shared memory and no synchronisation in the loop (the shared-memory
// version this replaces took ~13 us per solve: it sat on the critical path of the apply kernel).
// out[0..DEG]: highest power first (np.polyfit order), written by lane N.
template <int DEG>
__device__ __forceinline__ void solve_series(const double* __restrict__ mom, long long min_count, double* out,
                                             int lane) {
    constexpr int N = DEG + 1;
    constexpr unsigned int FULL = 0xffffffffu;
    const double count = mom[0];
    if (!(count >= (double)min_count)) {  // identity: poly_regression.py:38-41
        if (lane < N) out[lane] = (lane == N - 2) ? 1.0 : 0.0;
        return;
    }
    const int j = lane < N ? lane : N;
    const double sj = j < N ? sqrt(mom[2 * j]) : 1.0;
    double a[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const double si = sqrt(mom[2 * i]);
        const double num = j < N ? mom[i + j] : mom[2 * DEG + 1 + i];
        a[i] = num / (si * sj);
    }
#pragma unroll
    for (int c = 0; c < N; ++c) {
        int piv = c;  // lane c searches its own column
        double best = fabs(a[c]);
#pragma unroll
        for (int r = c + 1; r < N; ++r) {
            const double v = fabs(a[r]);
            if (v > best) {
                best = v;
                piv = r;
            }
        }
        piv = __shfl_sync(FULL, piv, c);
#pragma unroll
        for (int r = c + 1; r < N; ++r)
            if (r == piv) {
                const double t = a[c];
                a[c] = a[r];
                a[r] = t;
            }
        const double inv = 1.0 / __shfl_sync(FULL, a[c], c);
        a[c] *= inv;
#pragma unroll
        for (int r = 0; r < N; ++r)
            if (r != c) {
                const double f = __shfl_sync(FULL, a[r], c);  // column c, read before lane c rewrites it
                a[r] = fma(-f, a[c], a[r]);
            }
    }
    // un-scale; np.polyfit order is highest power first
    if (lane == N) {
#pragma unroll
        for (int i = 0; i < N; ++i) out[DEG - i] = a[i] / sqrt(mom[2 * i]);
    }
}

template <int DEG>
__global__ void __launch_bounds__(128) poly_solve_kernel(const double* __restrict__ moments, int K,
                                                         long long min_count, double* __restrict__ coeffs) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = blockIdx.x * 4 + w;
    if (k >= K) return;
    solve_series<DEG>(moments + (long long)k * (3 * DEG + 2), min_count, coeffs + (long long)k * (DEG + 1), lane);
}

template <int DEG>
__device__ __forceinline__ float horner_clip(float xf, const double (&c)[DEG + 1], bool use, float lo, float hi) {
    float r = xf;
    if (use) {
        const double x = (double)xf;
        double acc = 0.0;  // np.polyval starts from zeros_like(x): 0*Inf = NaN is kept
#pragma unroll
        for (int j = 0; j <= DEG; ++j) acc = fma(acc, x, c[j]);
        r = (float)acc;
    }
    if (lo <= hi) r = r < lo ? lo : (r > hi ? hi : r);  // NaN compares false twice and survives, as np.clip
    return r;
}

// np.polyval evaluates Horner as y = y*x + c (mul then add, two roundings); an fma differs
// by < 1 ulp of fp64, far below the fp32 result's resolution.
template <int DEG>
__global__ void __launch_bounds__(256) poly_apply_kernel(const float* __restrict__ x, long long x_k_stride,
                                                         long long x_n_stride, const double* __restrict__ coeffs,
                                                         const uint8_t* __restrict__ mask, long long mask_k_div,
                                                         long long mask_k_mod, long long n, float lo, float hi,
                                                         float* __restrict__ out,
                                                         long long out_k_stride, long long out_n_stride) {
    const int k = blockIdx.y;
    const float* xk = x + (long long)k * x_k_stride;
    float* ok = out + (long long)k * out_k_stride;
    const uint8_t* mk = mask ? mask + (((long long)k / mask_k_div) % mask_k_mod) * n : nullptr;
    double c[DEG + 1];
#pragma unroll
    for (int j = 0; j <= DEG; ++j) c[j] = coeffs[(long long)k * (DEG + 1) + j];

    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const bool vec = x_n_stride == 1 && out_n_stride == 1 &&
                     ((reinterpret_cast<uintptr_t>(xk) | reinterpret_cast<uintptr_t>(ok)) & 15) == 0 &&
                     (mk == nullptr || (reinterpret_cast<uintptr_t>(mk) & 3) == 0);
    long long done = 0;
    if (vec) {
        const long long n4 = n >> 2;
        const float4* x4 = reinterpret_cast<const float4*>(xk);
        float4* o4 = reinterpret_cast<float4*>(ok);
        const uchar4* m4 = reinterpret_cast<const uchar4*>(mk);
        for (long long i = tid; i < n4; i += nthreads) {
            const float4 xv = __ldg(x4 + i);
            uchar4 mv = make_uchar4(1, 1, 1, 1);
            if (mk) mv = __ldg(m4 + i);
            float4 r;
            r.x = horner_clip<DEG>(xv.x, c, mv.x != 0, lo, hi);
            r.y = horner_clip<DEG>(xv.y, c, mv.y != 0, lo, hi);
            r.z = horner_clip<DEG>(xv.z, c, mv.z != 0, lo, hi);
            r.w = horner_clip<DEG>(xv.w, c, mv.w != 0, lo, hi);
            o4[i] = r;
        }
        done = n4 << 2;
    }
    for (long long i = done + tid; i < n; i += nthreads) {
        const float xv = __ldg(xk + i * x_n_stride);
        ok[i * out_n_stride] = horner_clip<DEG>(xv, c, mk == nullptr || mk[i] != 0, lo, hi);
    }
}

// mask[g, i] = valid[g, i] && all_k finite(x[k, g, i]) && x[gate_k, g, i] > gate_gt   (poly_regression.py:106)
//              [&& all_k finite(y[k, g, i]) when y is given: `valid60 &= isfinite(s2_real_60m).all(0)`, :118]
// One thread per 4 pixels (16-byte loads when the planes allow it), grid = (blocks, G).
struct MaskParams {
    const float* x;
    long long xks, xgs;
    const float* y;  // nullable
    long long yks, ygs;
    const uint8_t* valid;  // nullable [G, n]
    uint8_t* mask;         // [G, n]
    long long n;
    int K, gate_k;
    float gate_gt;
    int vecx, vecy, vecm;
};

__device__ __forceinline__ float4 load4(const float* __restrict__ p, long long i, long long n, bool vec) {
    if (vec) return __ldg(reinterpret_cast<const float4*>(p + i));
    const float qnan = __int_as_float(0x7fc00000);  // out of range: not finite
    float4 r;
    r.x = (i + 0 < n) ? __ldg(p + i + 0) : qnan;
    r.y = (i + 1 < n) ? __ldg(p + i + 1) : qnan;
    r.z = (i + 2 < n) ? __ldg(p + i + 2) : qnan;
    r.w = (i + 3 < n) ? __ldg(p + i + 3) : qnan;
    return r;
}

__device__ __forceinline__ unsigned int finite_bits(const float4 v) {
    return (finite_f32(v.x) ? 1u : 0u) | (finite_f32(v.y) ? 2u : 0u) | (finite_f32(v.z) ? 4u : 0u) |
           (finite_f32(v.w) ? 8u : 0u);
}

__global__ void __launch_bounds__(256) fit_mask_kernel(const MaskParams P) {
    const long long g = blockIdx.y, n = P.n;
    const float* xg = P.x + g * P.xgs;
    const float* yg = P.y ? P.y + g * P.ygs : nullptr;
    const uint8_t* vg = P.valid ? P.valid + g * n : nullptr;
    uint8_t* mg = P.mask + g * n;
    const long long n4 = (n + 3) >> 2;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n4; q += (long long)gridDim.x * blockDim.x) {
        const long long i = q << 2;
        const bool full = i + 4 <= n;
        unsigned int m = 0xfu;
        if (vg) {
            if (full && P.vecm) {
                const uchar4 u = __ldg(reinterpret_cast<const uchar4*>(vg + i));
                m = (u.x ? 1u : 0u) | (u.y ? 2u : 0u) | (u.z ? 4u : 0u) | (u.w ? 8u : 0u);
            } else {
                m = 0u;
                for (int j = 0; j < 4; ++j)
                    if (i + j < n && vg[i + j]) m |= 1u << j;
            }
        }
        for (int k = 0; k < P.K; ++k) {
            const float4 v = load4(xg + (long long)k * P.xks, i, n, full && P.vecx);
            m &= finite_bits(v);
            if (k == P.gate_k)
                m &= (v.x > P.gate_gt ? 1u : 0u) | (v.y > P.gate_gt ? 2u : 0u) | (v.z > P.gate_gt ? 4u : 0u) |
                     (v.w > P.gate_gt ? 8u : 0u);
            if (yg) m &= finite_bits(load4(yg + (long long)k * P.yks, i, n, full && P.vecy));
        }
        if (full && P.vecm) {
            *reinterpret_cast<uchar4*>(mg + i) = make_uchar4(m & 1u, (m >> 1) & 1u, (m >> 2) & 1u, (m >> 3) & 1u);
        } else {
            for (int j = 0; j < 4; ++j)
                if (i + j < n) mg[i + j] = (m >> j) & 1u;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// (80 registers — three blocks per SM — keep the solve and the Horner coefficients of degree <= 5 in registers; the
// 64-register cap of round 1 spilled 16 bytes at degree 2 and 108-156 at the reference script's degree 4.)
// Fused solve + apply: grid = (blocks per series, S series).  Every thread first issues its first
// batch of loads, THEN warp 0 solves the block's series (a 3 x 3 system for degree 2: cheaper than a
// launch, and hidden behind the DRAM latency of the loads already in flight); the block then maps its
// share of the samples (Horner in fp64, mask, clip: poly_regression.py:65-84), four 16-byte loads in
// flight per thread.  Optional percentile stretch of x first (s2_emit/color.py:25-34).
struct ApplyParams {
    const float* x;
    long long xks, xgs;  // series s = k * G + g  ->  x + k * xks + g * xgs
    float* out;
    long long oks, ogs;
    const uint8_t* mask;  // nullable, [G, n]
    const double* moments;  // [S, 3*deg+2]
    const double* xst;      // nullable [S][2] (lo, hi) percentile stretch of x
    double* coeffs;         // [S, deg+1] (written by block x == 0 of every series)
    long long n, min_count;
    int G, vec;
    float lo, hi;
    Exchange ex;            // nranks > 1: the moments are the rank-ordered sum of the peer slots (and `moments` is
    double* moments_out;    // ignored); the sums are written here (nullable) by block x == 0 of every series
};

constexpr int APPLY_UNROLL = 2;

template <int DEG, bool STRETCH>
__global__ void __launch_bounds__(256, DEG <= 2 ? 4 : (DEG <= 5 ? 3 : 2)) solve_apply_kernel(const ApplyParams P) {
    __shared__ double cs[MAXDEG + 1];
    __shared__ double msum[3 * MAXDEG + 2];
    const int s = blockIdx.y;
    const int k = s / P.G, g = s - k * P.G;
    const float* xs = P.x + (long long)k * P.xks + (long long)g * P.xgs;
    float* os = P.out + (long long)k * P.oks + (long long)g * P.ogs;
    const uint8_t* mg = P.mask ? P.mask + (long long)g * P.n : nullptr;
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long n4 = P.vec ? (P.n >> 2) : 0;
    const float4* x4 = reinterpret_cast<const float4*>(xs);
    float4* o4 = reinterpret_cast<float4*>(os);
    const uchar4* m4 = reinterpret_cast<const uchar4*>(mg);
    constexpr bool stretch = STRETCH;
    double slo = 0.0, sden = 1.0, srcp = 1.0;
    if (stretch) {
        slo = P.xst[2 * (long long)s];
        sden = P.xst[2 * (long long)s + 1] - slo + 1e-12;
        srcp = 1.0 / sden;
    }

    // two register buffers of APPLY_UNROLL 16-byte loads: the next batch is requested before the current one is
    // mapped and stored, so 2 * APPLY_UNROLL loads per thread are in flight throughout
    float4 xa[APPLY_UNROLL], xb[APPLY_UNROLL];
    uchar4 ma[APPLY_UNROLL], mb[APPLY_UNROLL];
    auto fetch = [&](long long i, float4 (&xv)[APPLY_UNROLL], uchar4 (&mv)[APPLY_UNROLL]) {
#pragma unroll
        for (int u = 0; u < APPLY_UNROLL; ++u) {
            const long long iu = i + u * nthreads;
            mv[u] = make_uchar4(1, 1, 1, 1);
            if (iu < n4) {
                xv[u] = __ldg(x4 + iu);
                if (mg) mv[u] = __ldg(m4 + iu);
            }
        }
    };
    const long long batch = APPLY_UNROLL * nthreads;
    long long i = tid;
    if (i < n4) fetch(i, xa, ma);  // in flight while warp 0 solves
    if (i + batch < n4) fetch(i + batch, xb, mb);

    if (threadIdx.x < 32) {
        const double* mom = P.moments + (long long)s * (3 * DEG + 2);
        bool peers_ok = true;
        if (P.ex.nranks > 1) {
            // wait until every rank's sums of this epoch have landed in my peer block, then add them in rank order
            constexpr int M = 3 * DEG + 2;
            // the epoch this rank published last (its finalize precedes this kernel on the stream)
            const unsigned long long epoch = P.ex.epoch ? P.ex.epoch : *(volatile unsigned long long*)&P.ex.mine->epoch;
            const int par = (int)(epoch & 1ull);
            bool arrived = true;
            if ((int)threadIdx.x < P.ex.nranks)
                arrived = wait_flag(&P.ex.mine->flags[par][threadIdx.x], epoch, P.ex.mine, P.ex.timeout_ns);
            peers_ok = __all_sync(0xffffffffu, arrived);
            if (threadIdx.x < M) {
                double t = 0.0;
                for (int q = 0; q < P.ex.nranks; ++q) t += __ldcg(&P.ex.mine->slots[par][q][s * M + threadIdx.x]);
                if (!peers_ok) t = __longlong_as_double(0x7ff8000000000000LL);
                msum[threadIdx.x] = t;
                if (blockIdx.x == 0 && P.moments_out) P.moments_out[(long long)s * M + threadIdx.x] = t;
            }
            __syncwarp();
            mom = msum;
        }
        solve_series<DEG>(mom, P.min_count, cs, threadIdx.x);
        __syncwarp();
        // a peer never showed up: the sums are not the global ones -> NaN coefficients (a NaN count would otherwise
        // take the identity branch), never a silent per-rank fit; the host finds HSR_PEER_TIMEOUT in the status word
        if (!peers_ok && threadIdx.x <= DEG) cs[threadIdx.x] = __longlong_as_double(0x7ff8000000000000LL);
        __syncwarp();
        if (blockIdx.x == 0 && threadIdx.x <= DEG) P.coeffs[(long long)s * (DEG + 1) + threadIdx.x] = cs[threadIdx.x];
    }
    __syncthreads();
    double c[DEG + 1];
#pragma unroll
    for (int j = 0; j <= DEG; ++j) c[j] = cs[j];

    auto map4 = [&](float4 v, uchar4 m) {
        if (stretch) v = stretch4(v, slo, sden, srcp);
        float4 r;
        r.x = horner_clip<DEG>(v.x, c, m.x != 0, P.lo, P.hi);
        r.y = horner_clip<DEG>(v.y, c, m.y != 0, P.lo, P.hi);
        r.z = horner_clip<DEG>(v.z, c, m.z != 0, P.lo, P.hi);
        r.w = horner_clip<DEG>(v.w, c, m.w != 0, P.lo, P.hi);
        return r;
    };
    auto flush = [&](long long i0, const float4 (&xv)[APPLY_UNROLL], const uchar4 (&mv)[APPLY_UNROLL]) {
#pragma unroll
        for (int u = 0; u < APPLY_UNROLL; ++u) {
            const long long iu = i0 + u * nthreads;
            if (iu < n4) __stcs(o4 + iu, map4(xv[u], mv[u]));
        }
    };
    while (i < n4) {
        flush(i, xa, ma);
        if (i + 2 * batch < n4) fetch(i + 2 * batch, xa, ma);
        i += batch;
        if (i >= n4) break;
        flush(i, xb, mb);
        if (i + 2 * batch < n4) fetch(i + 2 * batch, xb, mb);
        i += batch;
    }
    for (long long e = (n4 << 2) + tid; e < P.n; e += nthreads) {
        float v = __ldg(xs + e);
        if (stretch) v = stretch1(v, slo, sden, srcp);
        os[e] = horner_clip<DEG>(v, c, mg == nullptr || mg[e] != 0, P.lo, P.hi);
    }
}

#define HSR_DEG_SWITCH(deg, CALL)  \
    switch (deg) {                 \
        case 1: CALL(1); break;    \
        case 2: CALL(2); break;    \
        case 3: CALL(3); break;    \
        case 4: CALL(4); break;    \
        case 5: CALL(5); break;    \
        case 6: CALL(6); break;    \
        case 7: CALL(7); break;    \
        default: CALL(8); break;   \
    }

// Grids are sized so that every block is resident at once (no tail wave): resident = SMs x the occupancy
// the runtime reports for the kernel; the blocks are dealt evenly to the S series.
// (the occupancy query is cached per kernel instantiation and device: `cache` is that instantiation's static)
#define HSR_RESIDENT(kern, threads) \
    ([]() -> int { static int cache__[HSR_MAX_DEVICES]; return resident_blocks_cached(kern, threads, cache__); }())

int blocks_per_series(long long n, long long S, int resident, long long px_per_block) {
    long long per = (n + px_per_block - 1) / px_per_block;
    if (per < 1) per = 1;
    long long cap = resident / (S > 0 ? S : 1);
    if (cap < 1) cap = 1;
    return (int)(per < cap ? per : cap);
}

int make_exchange(const hsr_exchange_t* e, long long doubles, Exchange* out) {
    *out = Exchange{};
    if (e == nullptr || e->nranks <= 1) return HSR_OK;
    HSR_REQUIRE(e->peer_blocks && e->my_block, HSR_EINVAL, "exchange: null peer_blocks / my_block");
    HSR_REQUIRE(e->nranks <= PEER_MAXR && e->rank >= 0 && e->rank < e->nranks, HSR_ERANGE,
                "exchange: rank %d of %d (at most %d ranks)", e->rank, e->nranks, PEER_MAXR);
    HSR_REQUIRE(doubles <= PEER_MAXD, HSR_ERANGE, "exchange: %lld moments per rank exceed the %d-double slot", doubles,
                PEER_MAXD);
    out->peers = reinterpret_cast<PeerBlock* const*>(e->peer_blocks);
    out->mine = reinterpret_cast<PeerBlock*>(e->my_block);
    out->nranks = e->nranks;
    out->rank = e->rank;
    out->epoch = e->epoch;
    out->timeout_ns = (unsigned long long)(e->timeout_ms ? e->timeout_ms : HSR_PEER_DEFAULT_TIMEOUT_MS) * 1000000ull;
    return HSR_OK;
}

int moments_resident(int deg, bool stretch) {
    int r = 148;
#define CALL(D) r = stretch ? HSR_RESIDENT((poly_moments_kernel<D, true>), MOM_THREADS) \
                            : HSR_RESIDENT((poly_moments_kernel<D, false>), MOM_THREADS)
    HSR_DEG_SWITCH(deg, CALL)
#undef CALL
    return r;
}

// The workspace is sized for the plain kernel; the stretch variant (more registers) never gets more blocks.
int moments_blocks(long long n, long long S, int deg, bool stretch) {
    const int plain = blocks_per_series(n, S, moments_resident(deg, false), (long long)MOM_THREADS * 8);
    if (!stretch) return plain;
    const int st = blocks_per_series(n, S, moments_resident(deg, true), (long long)MOM_THREADS * 8);
    return st < plain ? st : plain;
}

int launch_moments(const MomParams& P, long long S, int deg, double* moments, cudaStream_t stream,
                   const Exchange& ex = Exchange{}) {
    const bool stretch = P.xst || P.yst;
    const int nblk = moments_blocks(P.n, S, deg, stretch);
    dim3 grid((unsigned int)nblk, (unsigned int)S);
#define CALL(D)                                                           \
    if (stretch)                                                          \
        poly_moments_kernel<D, true><<<grid, MOM_THREADS, 0, stream>>>(P); \
    else                                                                  \
        poly_moments_kernel<D, false><<<grid, MOM_THREADS, 0, stream>>>(P)
    HSR_DEG_SWITCH(deg, CALL)
#undef CALL
    HSR_CUDA(cudaGetLastError());
    moments_finalize_kernel<<<(unsigned int)S, 256, 0, stream>>>(P.partial, nblk, n_moments(deg), moments, ex);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

template <int DEG>
void launch_apply(const float* x, long long xks, long long xns, const double* coeffs, const uint8_t* mask,
                  long long mdiv, long long mmod, long long n, int K, float lo, float hi, float* out, long long oks,
                  long long ons, cudaStream_t stream) {
    const int nblk = blocks_per_series(n, K, HSR_RESIDENT(poly_apply_kernel<DEG>, 256), 256 * 8);
    dim3 grid((unsigned int)nblk, (unsigned int)K);
    poly_apply_kernel<DEG><<<grid, 256, 0, stream>>>(x, xks, xns, coeffs, mask, mdiv, mmod, n, lo, hi, out, oks,
                                                     ons);
}

}  // namespace

size_t poly_moments_workspace(long long n, int K, int deg) {
    if (n < 0 || K < 1 || deg < 1 || deg > MAXDEG) return 0;
    return (size_t)moments_blocks(n, K, deg, false) * (size_t)K * (size_t)n_moments(deg) * sizeof(double);
}

int poly_moments_impl(const float* x, long long xks, long long xns, const float* y, long long yks, long long yns,
                      const uint8_t* mask, long long mask_k_div, long long mask_k_mod, long long n, int K, int deg,
                      double* partial, double* moments, cudaStream_t stream) {
    HSR_REQUIRE(x && y && partial && moments, HSR_EINVAL, "null x / y / partial / moments pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && K <= 65535, HSR_EINVAL, "bad n = %lld or K = %d", n, K);
    HSR_REQUIRE(deg >= 1 && deg <= MAXDEG, HSR_ERANGE, "deg = %d outside [1, %d]", deg, MAXDEG);
    HSR_REQUIRE(mask == nullptr || (mask_k_div >= 1 && mask_k_mod >= 1), HSR_EINVAL,
                "mask_k_div / mask_k_mod must be >= 1");
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 3) == 0, HSR_EALIGN,
                "x / y not 4-byte aligned");
    MomParams P{};
    P.x = x, P.xks = xks, P.xgs = 0, P.xns = xns, P.y = y, P.yks = yks, P.ygs = 0, P.yns = yns;
    P.mask = mask, P.mdiv = mask ? mask_k_div : 1, P.mmod = mask ? mask_k_mod : 1;
    P.n = n, P.G = 1, P.partial = partial;
    return launch_moments(P, K, deg, moments, stream);
}

int poly_solve_impl(const double* moments, int K, int deg, long long min_count, double* coeffs, cudaStream_t stream) {
    HSR_REQUIRE(moments && coeffs, HSR_EINVAL, "null moments / coeffs pointer");
    HSR_REQUIRE(K >= 1, HSR_EINVAL, "K = %d", K);
    HSR_REQUIRE(deg >= 1 && deg <= MAXDEG, HSR_ERANGE, "deg = %d outside [1, %d]", deg, MAXDEG);
#define CALL(D) poly_solve_kernel<D><<<(unsigned int)((K + 3) / 4), 128, 0, stream>>>(moments, K, min_count, coeffs)
    HSR_DEG_SWITCH(deg, CALL)
#undef CALL
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int poly_apply_impl(const float* x, long long xks, long long xns, const double* coeffs, const uint8_t* mask,
                    long long mask_k_div, long long mask_k_mod, long long n, int K, int deg, float lo, float hi,
                    float* out, long long oks, long long ons, cudaStream_t stream) {
    HSR_REQUIRE(x && coeffs && out, HSR_EINVAL, "null x / coeffs / out pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && K <= 65535, HSR_EINVAL, "bad n = %lld or K = %d", n, K);
    HSR_REQUIRE(deg >= 1 && deg <= MAXDEG, HSR_ERANGE, "deg = %d outside [1, %d]", deg, MAXDEG);
    HSR_REQUIRE(mask == nullptr || (mask_k_div >= 1 && mask_k_mod >= 1), HSR_EINVAL,
                "mask_k_div / mask_k_mod must be >= 1");
    if (n == 0) return HSR_OK;
#define CALL(D) launch_apply<D>(x, xks, xns, coeffs, mask, mask_k_div, mask_k_mod, n, K, lo, hi, out, oks, ons, stream)
    HSR_DEG_SWITCH(deg, CALL)
#undef CALL
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int fit_mask_impl(const float* x, long long xks, long long xgs, const float* y, long long yks, long long ygs,
                  long long n, int K, int G, const uint8_t* valid, int gate_k, float gate_gt, uint8_t* mask,
                  cudaStream_t stream) {
    HSR_REQUIRE(x && mask, HSR_EINVAL, "null x / mask pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && G >= 1 && G <= 65535, HSR_EINVAL, "bad n = %lld, K = %d or G = %d", n, K, G);
    HSR_REQUIRE(gate_k < K, HSR_EINVAL, "gate_k = %d >= K = %d", gate_k, K);
    if (n == 0) return HSR_OK;
    MaskParams P{};
    P.x = x, P.xks = xks, P.xgs = xgs, P.y = y, P.yks = yks, P.ygs = ygs, P.valid = valid, P.mask = mask;
    P.n = n, P.K = K, P.gate_k = gate_k, P.gate_gt = gate_gt;
    const long long xs_or = (K > 1 ? xks : 0) | (G > 1 ? xgs : 0), ys_or = (K > 1 ? yks : 0) | (G > 1 ? ygs : 0);
    P.vecx = ((reinterpret_cast<uintptr_t>(x) | (uintptr_t)(xs_or * 4)) & 15) == 0 ? 1 : 0;
    P.vecy = ((reinterpret_cast<uintptr_t>(y) | (uintptr_t)(ys_or * 4)) & 15) == 0 ? 1 : 0;
    P.vecm = ((reinterpret_cast<uintptr_t>(valid) | reinterpret_cast<uintptr_t>(mask) | (uintptr_t)(G > 1 ? n : 0)) & 3) == 0
                 ? 1 : 0;
    const int nblk = blocks_per_series(n, G, HSR_RESIDENT(fit_mask_kernel, 256), 256 * 4);
    dim3 grid((unsigned int)nblk, (unsigned int)G);
    fit_mask_kernel<<<grid, 256, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

// Fit of the pair-synthesis pass: [fit mask unless it is given] -> moments of the K*G series.
int fit_moments_impl(const float* x, long long xks, long long xgs, const float* y, long long yks, long long ygs,
                     const uint8_t* valid, long long n, int K, int G, int deg, int gate_k, float gate_gt, int flags,
                     const double* x_stretch, const double* y_stretch, uint8_t* mask, double* partial,
                     double* moments, const hsr_exchange_t* exchange, cudaStream_t stream) {
    HSR_REQUIRE(x && y && partial && moments, HSR_EINVAL, "null x / y / partial / moments pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && K <= 65535, HSR_ERANGE, "bad n = %lld or K = %d", n, K);
    Exchange ex{};
    {
        const int rc = make_exchange(exchange, (long long)K * G * n_moments(deg), &ex);
        if (rc != HSR_OK) return rc;
    }
    HSR_REQUIRE(G >= 1 && (long long)K * G <= 65535, HSR_ERANGE, "K * G = %lld outside [1, 65535]", (long long)K * G);
    HSR_REQUIRE(deg >= 1 && deg <= MAXDEG, HSR_ERANGE, "deg = %d outside [1, %d]", deg, MAXDEG);
    HSR_REQUIRE(gate_k < K, HSR_EINVAL, "gate_k = %d >= K = %d", gate_k, K);
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 3) == 0, HSR_EALIGN,
                "x / y not 4-byte aligned");
    const uint8_t* fm = valid;
    if (flags & HSR_FIT_MASK_GIVEN) {
        HSR_REQUIRE(valid, HSR_EINVAL, "HSR_FIT_MASK_GIVEN needs the mask in `valid`");
    } else {
        HSR_REQUIRE(mask, HSR_EINVAL, "null mask pointer (the fit mask is an output unless HSR_FIT_MASK_GIVEN)");
        int rc = fit_mask_impl(x, xks, xgs, (flags & HSR_FIT_Y_FINITE) ? y : nullptr, yks, ygs, n, K, G, valid, gate_k,
                               gate_gt, mask, stream);
        if (rc != HSR_OK) return rc;
        fm = mask;
    }
    MomParams P{};
    P.x = x, P.xks = xks, P.xgs = xgs, P.xns = 1, P.y = y, P.yks = yks, P.ygs = ygs, P.yns = 1;
    P.mask = fm, P.mdiv = 1, P.mmod = G;  // series s = k * G + g uses mask row g
    P.xst = x_stretch, P.yst = y_stretch;
    P.n = n, P.G = G, P.partial = partial;
    P.reverse = 1;
    return launch_moments(P, (long long)K * G, deg, moments, stream, ex);
}

int moments_sum_impl(const double* per_unit, int units, long long count, double* out, const hsr_exchange_t* exchange,
                     cudaStream_t stream) {
    HSR_REQUIRE(out && (per_unit || units == 0), HSR_EINVAL, "null per_unit / out pointer");
    HSR_REQUIRE(units >= 0 && count >= 1, HSR_EINVAL, "bad units = %d or count = %lld", units, count);
    Exchange ex{};
    {
        const int rc = make_exchange(exchange, count, &ex);
        if (rc != HSR_OK) return rc;
    }
    moments_sum_kernel<<<(unsigned int)((count + 255) / 256), 256, 0, stream>>>(per_unit, units, count, out, ex);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

size_t fit_moments_workspace(long long n, int K, int G, int deg) {
    if (n < 0 || K < 1 || G < 1 || deg < 1 || deg > MAXDEG) return 0;
    return (size_t)moments_blocks(n, (long long)K * G, deg, false) * (size_t)K * (size_t)G * (size_t)n_moments(deg) *
           sizeof(double);
}

int poly_solve_apply_impl(const float* x, long long xks, long long xgs, const double* moments, const uint8_t* mask,
                          long long n, int K, int G, int deg, long long min_count, float lo, float hi,
                          const double* x_stretch, double* coeffs, float* out, long long oks, long long ogs,
                          const hsr_exchange_t* exchange, double* moments_out, cudaStream_t stream) {
    HSR_REQUIRE(x && moments && coeffs && out, HSR_EINVAL, "null x / moments / coeffs / out pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && G >= 1 && (long long)K * G <= 65535, HSR_ERANGE,
                "bad n = %lld, K = %d or G = %d (K * G <= 65535)", n, K, G);
    HSR_REQUIRE(deg >= 1 && deg <= MAXDEG, HSR_ERANGE, "deg = %d outside [1, %d]", deg, MAXDEG);
    ApplyParams P{};
    P.x = x, P.xks = xks, P.xgs = xgs, P.out = out, P.oks = oks, P.ogs = ogs, P.mask = mask, P.moments = moments;
    P.coeffs = coeffs, P.n = n, P.min_count = min_count, P.G = G, P.lo = lo, P.hi = hi, P.xst = x_stretch;
    P.moments_out = moments_out;
    {
        const int rc = make_exchange(exchange, (long long)K * G * n_moments(deg), &P.ex);
        if (rc != HSR_OK) return rc;
    }
    const long long s_or = (K > 1 ? (xks | oks) : 0) | (G > 1 ? (xgs | ogs) : 0);  // strides that are stepped
    const uintptr_t a16 = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | (uintptr_t)(s_or * 4);
    const uintptr_t a4 = reinterpret_cast<uintptr_t>(mask) | (uintptr_t)(G > 1 ? n : 0);
    P.vec = ((a16 & 15) == 0 && (a4 & 3) == 0) ? 1 : 0;
    const long long S = (long long)K * G;
    int resident = 148;
#define CALL(D) resident = x_stretch ? HSR_RESIDENT((solve_apply_kernel<D, true>), 256) \
                                     : HSR_RESIDENT((solve_apply_kernel<D, false>), 256)
    HSR_DEG_SWITCH(deg, CALL)
#undef CALL
    const int nblk = blocks_per_series(n, S, resident, 256 * 4 * APPLY_UNROLL * 2);
    dim3 grid((unsigned int)nblk, (unsigned int)S);
#define CALL(D)                                                   \
    if (x_stretch)                                                \
        solve_apply_kernel<D, true><<<grid, 256, 0, stream>>>(P); \
    else                                                          \
        solve_apply_kernel<D, false><<<grid, 256, 0, stream>>>(P)
    HSR_DEG_SWITCH(deg, CALL)
#undef CALL
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

// ---- peer blocks and CUDA IPC plumbing (one block per rank, created once per process group)
size_t peer_block_bytes() { return sizeof(PeerBlock); }

int peer_alloc_impl(void** dptr) {
    HSR_REQUIRE(dptr, HSR_EINVAL, "null output pointer");
    HSR_CUDA(cudaMalloc(dptr, sizeof(PeerBlock)));
    HSR_CUDA(cudaMemset(*dptr, 0, sizeof(PeerBlock)));
    HSR_CUDA(cudaDeviceSynchronize());
    return HSR_OK;
}

int peer_free_impl(void* dptr) {
    if (dptr) HSR_CUDA(cudaFree(dptr));
    return HSR_OK;
}

// Status word of this rank's block (sticky): synchronises `stream`, then reads it back.
int peer_status_impl(const void* dptr, unsigned int* status, cudaStream_t stream) {
    HSR_REQUIRE(dptr && status, HSR_EINVAL, "null pointer");
    HSR_CUDA(cudaStreamSynchronize(stream));
    const PeerBlock* b = reinterpret_cast<const PeerBlock*>(dptr);
    HSR_CUDA(cudaMemcpy(status, &b->error, sizeof(unsigned int), cudaMemcpyDeviceToHost));
    if (*status & HSR_PEER_TIMEOUT) {
        set_error("peer exchange timed out: a rank did not publish its moments (dead peer, or ranks ran different "
                  "numbers of exchanges); coefficients of that step are NaN");
        return HSR_EPEER;
    }
    return HSR_OK;
}

int ipc_export_impl(const void* dptr, unsigned char* handle) {
    HSR_REQUIRE(dptr && handle, HSR_EINVAL, "null pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == HSR_IPC_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    HSR_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(dptr)));
    memcpy(handle, &h, sizeof(h));
    return HSR_OK;
}

int ipc_import_impl(const unsigned char* handle, void** dptr) {
    HSR_REQUIRE(handle && dptr, HSR_EINVAL, "null pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    HSR_CUDA(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return HSR_OK;
}

int ipc_close_impl(void* dptr) {
    if (dptr) HSR_CUDA(cudaIpcCloseMemHandle(dptr));
    return HSR_OK;
}

}  // namespace hsr
