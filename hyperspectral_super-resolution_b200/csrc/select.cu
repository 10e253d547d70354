// select.cu — shared percentile stretch (SURVEY section 8f row 1): exact masked percentiles of fp32 planes (sampled
// brackets + one streaming pass + an exact finish), and the stretch itself.
//
// Reference: s2_emit/color.py:25-34 (apply_shared_percentile_stretch), called between the SRF synthesis and
// the polynomial fit at s2_emit/poly_regression.py:126-127:
//     vals = img[..., c][mask];  lo, hi = np.percentile(vals, [pmin, pmax])
//     out[..., c] = np.clip((img[..., c] - lo) / (hi - lo + 1e-12), 0, 1)          (float64 -> float32)
// np.percentile (method "linear") on n masked samples: virtual index v = (n - 1) * q/100, neighbours
// a = sorted[floor(v)], b = sorted[floor(v) + 1] (both the last element when v >= n - 1), gamma = v - floor(v),
// result = a + (b - a) * gamma, or b - (b - a) * (1 - gamma) when gamma >= 0.5, with b - a rounded in fp32 and
// the rest in fp64; NaN anywhere among the samples makes every percentile NaN.  All of that is reproduced
// bit for bit: the order statistics are found exactly (the sample only chooses where to look), the interpolation
// follows numpy's operation order with explicitly un-fused fp64 arithmetic.
//
// Selection in THREE launches and ONE pass over the planes (r1: 8 launches, 3 passes; VERDICT r1 item 4).  Keys are
// the usual order-preserving u32 image of fp32 (-0 folded onto +0, NaNs counted apart).
//   1. select_sample_kernel (one block per series): a strided sample of <= 8192 masked samples goes to shared memory;
//      for every percentile the block finds, by a radix select over the sample, two sample keys that BRACKET the
//      order statistics wanted — the sample quantile -/+ 5 standard deviations of its rank.  Small series (n <= 8192)
//      are sampled completely; series whose sample holds < 64 masked values get the bracket [0, 2^32).
//   2. select_collect_kernel (the streaming pass, all SMs): every masked sample is compared with its series'
//      brackets: counted if below, equal to the lower key or equal to the upper key (ties at the bracket's ends — e.g.
//      a clipped image's 10 % of exact zeros — cost nothing), APPENDED to the bracket's candidate list if strictly
//      inside (~1 % of the samples).  Also the exact masked / NaN counts numpy's ranks need.
//   3. select_finish_kernel (one block per series): ranks r0 = floor((n - 1) q), r1 = r0 + 1 as numpy forms them;
//      located among {below, == lower key, candidates, == upper key}; ranks that fall among the candidates are found
//      by a radix select over the list in shared memory; interpolation in numpy's operation order.
// EXACT in every case: if a bracket misses its rank or the candidates overflow (adversarial distributions), the block
// falls back to a radix select over the whole series from global memory — slow (one SM reads the series four times)
// but never wrong, and it does not happen on image-like data.
#include <math.h>

#include "hsr_common.cuh"

namespace hsr {

namespace {

constexpr int SEL_QMAX = HSR_MAX_PERCENTILES;
constexpr int SEL_SAMPLE = 8192;      // samples per series in the bracket search
constexpr int SEL_CAP = 49152;        // candidates per bracket the finish kernel can hold (192 KB of shared memory)
constexpr int SEL_BT = 1024;          // threads of the sample / finish kernels
constexpr int SEL_THREADS = 256;      // threads of the streaming pass
constexpr int SEL_MAXR = 2 * SEL_QMAX;

struct SelSeries {
    unsigned int klo[SEL_QMAX], khi[SEL_QMAX];      // bracket keys (klo <= khi)
    unsigned int ncand[SEL_QMAX];                    // candidates appended (may exceed the capacity: overflow)
    unsigned int fell_back;                          // diagnostics: the finish kernel had to select over the whole series
    unsigned long long lt[SEL_QMAX], eqlo[SEL_QMAX], eqhi[SEL_QMAX];
    unsigned long long count, nan;                   // masked samples (NaNs included) and NaNs among them
};
static_assert(sizeof(SelSeries) == 96, "tests/test_gpu_select_paths.py and profiles/prof_select.py read this layout");

struct SelParams {
    const float* x[2];     // one or two plane sets (x planes, y planes); series s: set = s / S1, k = (s % S1) / G, g = s % G
    long long xks[2], xgs[2];
    int vec[2];
    int nsets;
    long long S1;          // series per set = K * G
    const uint8_t* mask;   // nullable [G, n]
    long long n;
    int G, Q;
    unsigned int cap;      // candidate capacity per bracket
    SelSeries* st;         // [nsets * S1]
    unsigned int* cand;    // [nsets * S1][Q][cap]
    const double* q;       // [Q] fractions
    double* out[2];        // [S1][Q] per set
};

__device__ __forceinline__ bool key_of(float v, unsigned int& key) {
    unsigned int u = __float_as_uint(v);
    if ((u & 0x7fffffffu) > 0x7f800000u) return false;  // NaN
    if ((u << 1) == 0u) u = 0u;                         // -0 -> +0 (equal under numpy's ordering)
    key = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return true;
}

__device__ __forceinline__ float value_of(unsigned int key) {
    const unsigned int u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
    return __uint_as_float(u);
}

struct SeriesRef {
    const float* xs;
    const uint8_t* mg;
    int vec;
};

__device__ __forceinline__ SeriesRef series_of(const SelParams& P, long long s) {
    const int set = (int)(s / P.S1);
    const long long ss = s - (long long)set * P.S1;
    const long long k = ss / P.G, g = ss - k * P.G;
    SeriesRef r;
    r.xs = P.x[set] + k * P.xks[set] + g * P.xgs[set];
    r.mg = P.mask ? P.mask + g * P.n : nullptr;
    r.vec = P.vec[set];
    return r;
}

// Block-wide simultaneous radix select (passes of 8 bits, most significant first): out[r] = the key of rank ranks[r]
// (0-based, ascending) among the keys `each` enumerates.  each(f) must call f(key, valid) the SAME number of times on
// every lane of a warp (invalid calls carry no key) and enumerate the same multiset every time it is called.  All the
// keys are known to share their bits above `nbits` (given as `common`): the passes cover the low nbits only — a narrow
// bracket's candidates differ in ~16 bits, and a pass over bits they all share would serialise every atomic on one
// bin.  A warp whose keys all fall into one bin adds 32 with one atomic.
// R <= SEL_MAXR <= number of warps.  All threads must call.
struct MultiSel {
    unsigned int hist[SEL_MAXR][256];
    unsigned int prefix[SEL_MAXR];
    unsigned long long rank[SEL_MAXR];
};

template <typename Each>
__device__ void block_multiselect(MultiSel& ms, int R, const unsigned long long* ranks, unsigned int* out, int nbits,
                                  unsigned int common, Each each) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int npass = (nbits + 7) / 8;                       // the passes cover the low 8 * npass >= nbits bits
    if (tid < R) {
        ms.prefix[tid] = 8 * npass >= 32 ? 0u : (common >> (8 * npass));
        ms.rank[tid] = ranks[tid];
    }
    for (int pass = 0; pass < npass; ++pass) {
        const int shift = 8 * (npass - 1 - pass);
        for (int i = tid; i < R * 256; i += blockDim.x) (&ms.hist[0][0])[i] = 0u;
        __syncthreads();
        unsigned int pre[SEL_MAXR];
#pragma unroll
        for (int r = 0; r < SEL_MAXR; ++r) pre[r] = r < R ? ms.prefix[r] : 0u;
        each([&](unsigned int key, bool valid) {
            const unsigned int hi = shift + 8 >= 32 ? 0u : (key >> (shift + 8));
            const unsigned int digit = (key >> shift) & 255u;
#pragma unroll
            for (int r = 0; r < SEL_MAXR; ++r) {
                if (r >= R) break;
                const bool hit = valid && (shift + 8 >= 32 || hi == pre[r]);
                const unsigned int tag = hit ? digit : 0xffffffffu;
                const unsigned int t0 = __shfl_sync(0xffffffffu, tag, 0);
                if (__all_sync(0xffffffffu, tag == t0)) {     // the whole warp in one bin (or nobody): one atomic
                    if (lane == 0 && t0 != 0xffffffffu) atomicAdd(&ms.hist[r][t0], 32u);
                } else if (hit) {
                    atomicAdd(&ms.hist[r][digit], 1u);
                }
            }
        });
        __syncthreads();
        if (warp < R) {     // warp r locates the bin of rank[r]: lane l owns bins 8 l .. 8 l + 7
            unsigned int c[8];
            unsigned long long local = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                c[j] = ms.hist[warp][lane * 8 + j];
                local += c[j];
            }
            unsigned long long incl = local;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            unsigned long long excl = incl - local;
            const unsigned long long rk = ms.rank[warp];
            if (rk >= excl && rk < excl + local) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (rk >= excl && rk < excl + c[j]) {
                        ms.prefix[warp] = (ms.prefix[warp] << 8) | (unsigned int)(lane * 8 + j);
                        ms.rank[warp] = rk - excl;
                    }
                    excl += c[j];
                }
            }
        }
        __syncthreads();
    }
    if (tid < R) out[tid] = ms.prefix[tid];
    __syncthreads();
}

// numpy's percentile ranks (method "linear") for n samples: virtual index (n - 1) q, neighbours floor / floor + 1,
// both the last element when the index is >= n - 1 (numpy then forms gamma from index -1)
__device__ __forceinline__ void numpy_ranks(long long n, double q, long long& r0, long long& r1, double& gamma) {
    const double vi = __dmul_rn((double)(n - 1), q);
    double prev = floor(vi);
    r0 = (long long)prev;
    r1 = r0 + 1;
    if (vi >= (double)(n - 1)) {
        r0 = r1 = n - 1;
        prev = -1.0;
    }
    if (vi < 0.0) {
        r0 = r1 = 0;
        prev = 0.0;
    }
    gamma = vi - prev;
}

// numpy's "linear" interpolation between the order statistics with keys ka <= kb: the float32 neighbour difference,
// then float64 without contraction, b - diff (1 - gamma) when gamma >= 0.5
__device__ __forceinline__ double numpy_lerp(unsigned int ka, unsigned int kb, double gamma) {
    const float a = value_of(ka), b = value_of(kb);
    const float diff = __fsub_rn(b, a);
    double r = __dadd_rn((double)a, __dmul_rn((double)diff, gamma));
    if (gamma >= 0.5) r = __dsub_rn((double)b, __dmul_rn((double)diff, __dsub_rn(1.0, gamma)));
    return r;
}

// ---- 1. brackets from a sample
__global__ void __launch_bounds__(SEL_BT) select_sample_kernel(const SelParams P) {
    __shared__ unsigned int sk[SEL_SAMPLE];
    __shared__ unsigned int mv_s;
    __shared__ MultiSel ms;
    __shared__ unsigned long long ranks[SEL_MAXR];
    __shared__ unsigned int found[SEL_MAXR];
    const long long s = blockIdx.x;
    const SeriesRef sr = series_of(P, s);
    SelSeries* st = P.st + s;
    const int tid = threadIdx.x, lane = tid & 31;
    const long long n = P.n;
    if (tid == 0) mv_s = 0u;
    __syncthreads();
    const long long m = n < SEL_SAMPLE ? n : SEL_SAMPLE;
    for (long long j0 = 0; j0 < m; j0 += SEL_BT) {        // warp-uniform trip count (ballots below)
        const long long j = j0 + tid;
        unsigned int key = 0u;
        bool ok = false;
        if (j < m) {
            const long long idx = (long long)(((unsigned __int128)j * (unsigned __int128)n) / (unsigned __int128)m);
            if (sr.mg == nullptr || sr.mg[idx] != 0) ok = key_of(__ldg(sr.xs + idx), key);
        }
        const unsigned int bal = __ballot_sync(0xffffffffu, ok);
        unsigned int base = 0u;
        if (lane == 0 && bal) base = atomicAdd(&mv_s, (unsigned int)__popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (ok) sk[base + __popc(bal & ((1u << lane) - 1u))] = key;
    }
    __syncthreads();
    const int mv = (int)mv_s;
    const int Q = P.Q;
    const bool wide = mv < 64;                              // too few masked samples to estimate anything: take everything
    if (!wide && tid < Q) {
        // the sample rank of the q-quantile is binomial: centre q (mv - 1), sigma sqrt(mv q (1 - q)); -/+ (5 sigma + 3)
        const double qq = P.q[tid];
        const double c = qq * (double)(mv - 1), sd = sqrt((double)mv * qq * (1.0 - qq));
        const double mg = 5.0 * sd + 3.0;
        double lo = floor(c - mg), hi = ceil(c + mg);
        lo = lo < 0.0 ? 0.0 : lo;
        hi = hi > (double)(mv - 1) ? (double)(mv - 1) : hi;
        ranks[2 * tid] = (unsigned long long)lo;
        ranks[2 * tid + 1] = (unsigned long long)hi;
    }
    __syncthreads();
    if (!wide) {
        block_multiselect(ms, 2 * Q, ranks, found, 32, 0u, [&](auto f) {
            for (int i0 = 0; i0 < mv; i0 += SEL_BT) {
                const int i = i0 + tid;
                f(i < mv ? sk[i] : 0u, i < mv);
            }
        });
    }
    if (tid < Q) {
        unsigned int klo = 0u, khi = 0xffffffffu;
        if (!wide) {
            klo = found[2 * tid];
            khi = found[2 * tid + 1];
            // a bracket that reaches the sample's extremes is opened to the end of the key range: the sample's
            // minimum / maximum are not the series'
            if (ranks[2 * tid] == 0ull) klo = 0u;
            if (ranks[2 * tid + 1] == (unsigned long long)(mv - 1)) khi = 0xffffffffu;
        }
        st->klo[tid] = klo;
        st->khi[tid] = khi;
        st->ncand[tid] = 0u;
        st->lt[tid] = st->eqlo[tid] = st->eqhi[tid] = 0ull;
    }
    if (tid == 0) {
        st->count = st->nan = 0ull;
        st->fell_back = 0u;
    }
}

// ---- 2. the streaming pass
__global__ void __launch_bounds__(SEL_THREADS) select_collect_kernel(const SelParams P) {
    const long long s = blockIdx.y;
    const SeriesRef sr = series_of(P, s);
    SelSeries* st = P.st + s;
    const int Q = P.Q;
    unsigned int klo[SEL_QMAX], khi[SEL_QMAX];
#pragma unroll
    for (int b = 0; b < SEL_QMAX; ++b) {
        klo[b] = b < Q ? st->klo[b] : 0xffffffffu;
        khi[b] = b < Q ? st->khi[b] : 0xffffffffu;
    }
    unsigned int* cand = P.cand + (size_t)s * SEL_QMAX * P.cap;
    const unsigned int cap = P.cap;
    // candidates are staged per block in shared memory and appended to the series' list with ONE global atomic per
    // block and bracket (30 000 atomics with return value on one address serialised the whole pass: 305 us)
    constexpr unsigned int SB = 1024;
    __shared__ unsigned int s_buf[SEL_QMAX][SB];
    __shared__ unsigned int s_n[SEL_QMAX], s_base[SEL_QMAX];
    if (threadIdx.x < SEL_QMAX) s_n[threadIdx.x] = 0u;
    __syncthreads();
    unsigned int cnt = 0, nan = 0, lt[SEL_QMAX] = {}, eqlo[SEL_QMAX] = {}, eqhi[SEL_QMAX] = {};
    // Common path per sample: is the sample masked, and does its key fall into the interval where its contribution is
    // known without looking at the brackets one by one?  With two ordered brackets (the 2 / 98 stretch) that interval is
    // (khi[0], klo[1]): such a sample is above bracket 0 and below bracket 1 — 96 % of the masked samples, three
    // instructions.  Everything else (inside or beyond a bracket, NaN, other bracket layouts) is revisited per batch of
    // 16 samples: one divergent detour per batch instead of one per sample.  Unmasked float4s are skipped whole.
    const bool fastiv = Q == 2 && khi[0] < klo[1];
    const unsigned int ivlo = fastiv ? khi[0] + 1u : 0u, ivlen = fastiv ? klo[1] - khi[0] - 1u : 0u;
    auto key_bits = [&](float v) -> unsigned int {          // order-preserving image of the float (-0 -> +0; NaNs beyond +-inf)
        unsigned int u = __float_as_uint(v);
        if ((u << 1) == 0u) u = 0u;
        return u ^ ((unsigned int)((int)u >> 31) | 0x80000000u);
    };
    auto detour = [&](unsigned int key) {                    // a masked sample outside the known interval
        if (key > 0xff800000u || key < 0x007fffffu) {        // NaN (positive / negative)
            ++nan;
            return;
        }
#pragma unroll
        for (int b = 0; b < SEL_QMAX; ++b) {
            if (b >= Q) break;
            if (key < klo[b]) {
                ++lt[b];
                continue;
            }
            if (key > khi[b]) continue;
            const bool atlo = key == klo[b], under = key < khi[b];
            eqlo[b] += atlo ? 1u : 0u;
            eqhi[b] += (!under && !atlo) ? 1u : 0u;
            if (!atlo && under) {
                const unsigned int sp = atomicAdd(&s_n[b], 1u);
                if (sp < SB) {
                    s_buf[b][sp] = key;
                } else {                                     // the block's buffer is full: straight to the list
                    const unsigned int pos = atomicAdd(&st->ncand[b], 1u);
                    if (pos < cap) cand[(size_t)b * cap + pos] = key;
                }
            }
        }
    };
    const long long n = P.n;
    const unsigned int tid = blockIdx.x * SEL_THREADS + threadIdx.x;
    const unsigned int nthreads = gridDim.x * SEL_THREADS;
    const unsigned int n4 = sr.vec ? (unsigned int)(n >> 2) : 0u;
    const float4* x4 = reinterpret_cast<const float4*>(sr.xs);
    const unsigned int* m4 = reinterpret_cast<const unsigned int*>(sr.mg);
    constexpr int UNR = 4;  // 16-byte loads in flight per thread
    // samples outside the known interval are queued per warp (ballot compaction) and revisited 32 at a time: at warp level
    // "rare per sample" is not rare (some lane of 32 needs the detour for 3 of 4 sample slots)
    __shared__ unsigned int s_q[SEL_THREADS / 32][64];
    unsigned int* wq = s_q[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const unsigned int lt_mask = (1u << lane) - 1u;
    unsigned int qn = 0u;                                    // queued keys of my warp (uniform)
    auto flush32 = [&]() {
        __syncwarp();
        const unsigned int key = wq[qn - 32u + lane];
        qn -= 32u;
        __syncwarp();
        detour(key);
    };
    for (unsigned int base0 = tid - lane; base0 < n4; base0 += UNR * nthreads) {   // warp-uniform trip count (ballots)
        const unsigned int base = base0 + lane;
        float4 v[UNR];
        unsigned int m[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const unsigned int i = base + u * nthreads;
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            m[u] = 0u;
            if (i < n4) {
                m[u] = sr.mg ? __ldg(m4 + i) : 0x01010101u;
                if (m[u]) v[u] = __ldcs(x4 + i);
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            if (__ballot_sync(0xffffffffu, m[u] != 0u) == 0u) continue;   // 128 unmasked samples (outside the swath: runs)
            const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const bool use = ((m[u] >> (8 * j)) & 0xffu) != 0u;
                const unsigned int key = key_bits(e[j]);
                const bool mid = use && (key - ivlo) < ivlen;
                cnt += use ? 1u : 0u;
                lt[SEL_QMAX - 1] += mid ? 1u : 0u;          // (fastiv implies Q == SEL_QMAX == 2: below bracket 1)
                const bool slow = use && !mid;
                const unsigned int bal = __ballot_sync(0xffffffffu, slow);
                if (bal) {
                    if (slow) wq[qn + __popc(bal & lt_mask)] = key;
                    qn += __popc(bal);
                    if (qn >= 32u) flush32();
                }
            }
        }
    }
    __syncwarp();
    if ((unsigned int)lane < qn) detour(wq[lane]);
    for (long long i = ((long long)n4 << 2) + tid; i < n; i += nthreads) {
        if (sr.mg != nullptr && sr.mg[i] == 0) continue;
        ++cnt;
        const unsigned int key = key_bits(__ldg(sr.xs + i));
        if ((key - ivlo) < ivlen) ++lt[SEL_QMAX - 1];
        else detour(key);
    }

    // the block's candidates -> the series' lists
    __syncthreads();
    if (threadIdx.x < Q) {
        const unsigned int nb = s_n[threadIdx.x] < SB ? s_n[threadIdx.x] : SB;
        s_n[threadIdx.x] = nb;
        s_base[threadIdx.x] = nb ? atomicAdd(&st->ncand[threadIdx.x], nb) : 0u;
    }
    __syncthreads();
    for (int b = 0; b < Q; ++b) {
        const unsigned int nb = s_n[b], base = s_base[b];
        for (unsigned int i = threadIdx.x; i < nb; i += SEL_THREADS)
            if (base + i < cap) cand[(size_t)b * cap + base + i] = s_buf[b][i];
    }
    // block totals -> the series' counters
    __shared__ unsigned long long red[SEL_THREADS / 32][2 + 3 * SEL_QMAX];
    const int warp = threadIdx.x >> 5;
    unsigned long long vals[2 + 3 * SEL_QMAX];
    vals[0] = cnt;
    vals[1] = nan;
#pragma unroll
    for (int b = 0; b < SEL_QMAX; ++b) {
        vals[2 + 3 * b] = lt[b];
        vals[3 + 3 * b] = eqlo[b];
        vals[4 + 3 * b] = eqhi[b];
    }
#pragma unroll
    for (int j = 0; j < 2 + 3 * SEL_QMAX; ++j) {
        unsigned long long v = vals[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][j] = v;
    }
    __syncthreads();
    if (threadIdx.x < 2 + 3 * SEL_QMAX) {
        unsigned long long t = 0;
#pragma unroll
        for (int w = 0; w < SEL_THREADS / 32; ++w) t += red[w][threadIdx.x];
        if (t) {
            unsigned long long* dst = threadIdx.x == 0 ? &st->count : threadIdx.x == 1 ? &st->nan
                                      : ((threadIdx.x - 2) % 3 == 0 ? &st->lt[(threadIdx.x - 2) / 3]
                                         : (threadIdx.x - 2) % 3 == 1 ? &st->eqlo[(threadIdx.x - 2) / 3]
                                                                      : &st->eqhi[(threadIdx.x - 2) / 3]);
            atomicAdd(dst, t);
        }
    }
}

// ---- 3. ranks -> order statistics -> percentiles: one block per (series, percentile)
__global__ void __launch_bounds__(SEL_BT) select_finish_kernel(const SelParams P) {
    extern __shared__ unsigned int ck[];                     // the bracket's candidates
    __shared__ MultiSel ms;
    __shared__ unsigned long long ranks[SEL_MAXR];
    __shared__ unsigned int found[SEL_MAXR];
    __shared__ unsigned int keys[2];                         // order statistics r0, r1
    __shared__ int how[2];                                   // 0 resolved, 1 among the candidates, 2 fall back
    __shared__ unsigned long long want[2], local[2];         // global ranks; ranks among the candidates
    __shared__ unsigned int red_lt[SEL_BT / 32], red_eq[SEL_BT / 32], red_next[SEL_BT / 32];
    const long long s = blockIdx.x;
    const int b = blockIdx.y;                                // my percentile
    const SeriesRef sr = series_of(P, s);
    const SelSeries* st = P.st + s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Q = P.Q;
    const int set = (int)(s / P.S1);
    double* out = P.out[set] + (s - (long long)set * P.S1) * Q + b;
    const long long n = (long long)st->count;
    if (n == 0 || st->nan != 0) {                            // no samples, or a NaN among them: every percentile is NaN
        if (tid == 0) *out = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    long long r0, r1;
    double gamma;
    numpy_ranks(n, P.q[b], r0, r1, gamma);
    // where do the two ranks fall: below the bracket (miss), == klo, candidates, == khi, above (miss)
    const unsigned long long lt = st->lt[b], eqlo = st->eqlo[b], eqhi = st->eqhi[b];
    const unsigned int nc = st->ncand[b];
    const unsigned int kl = st->klo[b], kh = st->khi[b];
    if (tid < 2) {
        unsigned long long r = (unsigned long long)(tid ? r1 : r0);
        want[tid] = r;
        int h = 2;
        if (r >= lt) {
            r -= lt;
            if (r < eqlo) {
                keys[tid] = kl;
                h = 0;
            } else {
                r -= eqlo;
                if (r < nc) {
                    h = nc <= P.cap ? 1 : 2;
                    local[tid] = r;
                } else {
                    r -= nc;
                    if (r < eqhi) {
                        keys[tid] = kh;
                        h = 0;
                    }
                }
            }
        }
        how[tid] = h;
    }
    __syncthreads();
    const int h0 = how[0], h1 = how[1];
    const bool fallback = h0 == 2 || h1 == 2;
    if (!fallback && (h0 == 1 || h1 == 1)) {
        const unsigned int* cg = P.cand + ((size_t)s * SEL_QMAX + b) * P.cap;
        for (unsigned int i = tid; i < nc; i += SEL_BT) ck[i] = cg[i];
        if (tid == 0) ranks[0] = h0 == 1 ? local[0] : local[1];
        __syncthreads();
        // the candidates lie strictly between klo and khi: they share the bits these two share
        const int nbits = 32 - __clz((int)(kl ^ kh));
        block_multiselect(ms, 1, ranks, found, nbits < 1 ? 1 : nbits, kl, [&](auto f) {
            for (unsigned int i0 = 0; i0 < nc; i0 += SEL_BT) {
                const unsigned int i = i0 + tid;
                f(i < nc ? ck[i] : 0u, i < nc);
            }
        });
        const unsigned int a = found[0];
        if (h0 == 1 && h1 == 1 && r1 != r0) {
            // r1 = r0 + 1: the same key if the candidates <= a reach past it, else the smallest candidate above a
            unsigned int c_le = 0u, nxt = 0xffffffffu;
            for (unsigned int i = tid; i < nc; i += SEL_BT) {
                const unsigned int k = ck[i];
                c_le += k <= a ? 1u : 0u;
                nxt = (k > a && k < nxt) ? k : nxt;
            }
            c_le = __reduce_add_sync(0xffffffffu, c_le);
            nxt = __reduce_min_sync(0xffffffffu, nxt);
            if (lane == 0) {
                red_eq[warp] = c_le;
                red_next[warp] = nxt;
            }
            __syncthreads();
            if (tid == 0) {
                unsigned int tot = 0u, mn = 0xffffffffu;
                for (int w = 0; w < SEL_BT / 32; ++w) {
                    tot += red_eq[w];
                    mn = red_next[w] < mn ? red_next[w] : mn;
                }
                keys[0] = a;
                keys[1] = local[1] < (unsigned long long)tot ? a : mn;
            }
        } else if (tid == 0) {
            if (h0 == 1) keys[0] = a;
            if (h1 == 1) keys[1] = a;                        // (h0 != 1, or r1 == r0: the one rank selected)
        }
        __syncthreads();
    }
    (void)red_lt;
    if (fallback) {
        // a bracket missed its rank or overflowed: radix select over the whole series (4 passes from global memory by
        // this one block) — slow, exact, and not expected on image-like data
        if (tid == 0) atomicAdd(&P.st[s].fell_back, 1u);
        const long long nn = P.n;
        block_multiselect(ms, 2, want, found, 32, 0u, [&](auto f) {
            for (long long i0 = 0; i0 < nn; i0 += SEL_BT) {
                const long long i = i0 + tid;
                unsigned int key = 0u;
                const bool ok = i < nn && (sr.mg == nullptr || sr.mg[i] != 0) && key_of(__ldg(sr.xs + i), key);
                f(key, ok);
            }
        });
        if (tid < 2) keys[tid] = found[tid];
    }
    __syncthreads();
    if (tid == 0) *out = numpy_lerp(keys[0], keys[1], gamma);
}

// ---- exact percentiles of a UNION of units (granules, slabs, ranks): radix select by 4 passes of 8 bits, most
// significant first.  Each pass every unit adds its counts to a per-series (pass 0) or per-target (passes 1-3) 256-bin
// histogram; the caller sums the histograms over its processes; a one-block-per-series step picks the digit of every
// target.  Only integer counts cross units and processes, and integer sums do not depend on the order they are formed
// in: every process ends with the same keys, and they are those of np.percentile over the concatenation.
//   state:  UnionSeries[S], then the u64 histograms [S][HS] the counting kernel accumulates into
//   hist:   the f64 image of the u64 histograms [S][HS] (exact below 2^53): what the processes all-reduce
// Series s of a unit: set s / K (0: x, 1: y), plane s % K.  Targets per series T = 2Q (ranks r0, r1 per percentile).
constexpr int UNI_THREADS = 256;
constexpr int UNI_UNR = 4;      // 16-byte loads in flight per thread

struct UnionSeries {
    unsigned long long rank[SEL_MAXR];   // target t: rank still to find among the keys that carry prefix[t]
    unsigned int prefix[SEL_MAXR];       // the key bits found so far (8 per pass)
    double gamma[SEL_QMAX];
    unsigned int dead;                   // NaN among the samples, no sample, or counts that do not add up: NaN results
    unsigned int ticket;                 // blocks of the running count launch that have finished this series
};

static_assert(sizeof(UnionSeries) == 72, "tests/test_gpu_union_select.py reads this layout");

struct UnionHead {
    double q[SEL_QMAX];                  // percentile fractions, copied by begin
};

__host__ __device__ constexpr int union_hist_stride(int Q) { return 2 * Q * 256 + 1; }   // + the NaN count (pass 0)

struct UnionCountParams {
    const float* x[2];
    long long xks[2];
    int vec[2];
    const uint8_t* mask;    // nullable [n]
    long long n;
    int K, S, Q, pass;
    UnionSeries* ser;
    unsigned long long* hu;
    double* hf;
};

// One streaming pass over one unit's planes: blockIdx.y = series.  Image data in [0, 1] has a handful of distinct top
// bytes, so a shared-memory atomic per sample would serialise on a few bins: the lanes of a warp that add to the same bin
// are grouped with __match_any_sync and their leader adds them with one atomic.
// NR: histograms per series of this pass (1 in pass 0, 2Q after it).
template <int NR>
__global__ void __launch_bounds__(UNI_THREADS) union_count_kernel(const UnionCountParams P) {
    __shared__ unsigned int h[NR][256];
    __shared__ unsigned int pre_s[NR];
    __shared__ unsigned int red[UNI_THREADS / 32];
    __shared__ int last;
    const int s = blockIdx.y;
    const int set = s / P.K, k = s - set * P.K;
    const float* xs = (set ? P.x[1] : P.x[0]) + (long long)k * (set ? P.xks[1] : P.xks[0]);   // (no dynamic param index)
    const int HS = union_hist_stride(P.Q);
    constexpr int R = NR;
    const int shift = 24 - 8 * P.pass;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool live = P.ser[s].dead == 0u;
    for (int i = tid; i < R * 256; i += UNI_THREADS) (&h[0][0])[i] = 0u;
    if (tid < R) pre_s[tid] = P.ser[s].prefix[tid];
    __syncthreads();
    unsigned int pre[R];
#pragma unroll
    for (int r = 0; r < R; ++r) pre[r] = pre_s[r];
    unsigned int nan = 0u;
    // every lane of the warp calls add() the same number of times (warp-uniform loops below)
    auto add = [&](float v, bool use) {
        unsigned int key = 0u;
        const bool ok = use && key_of(v, key);
        nan += (use && !ok) ? 1u : 0u;
        const unsigned int digit = (key >> shift) & 255u;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const bool hit = ok && (NR == 1 || (key >> (shift + 8)) == pre[r]);
            if (__ballot_sync(0xffffffffu, hit) == 0u) continue;
            const unsigned int peers = __match_any_sync(0xffffffffu, hit ? digit : 0x100u);
            if (hit && lane == __ffs(peers) - 1) atomicAdd(&h[r][digit], (unsigned int)__popc(peers));
        }
    };
    if (live) {
        const long long n = P.n;
        const long long gtid = (long long)blockIdx.x * UNI_THREADS + tid;
        const long long nthreads = (long long)gridDim.x * UNI_THREADS;
        const long long n4 = (set ? P.vec[1] : P.vec[0]) ? (n >> 2) : 0;
        const float4* x4 = reinterpret_cast<const float4*>(xs);
        const unsigned int* m4 = reinterpret_cast<const unsigned int*>(P.mask);
        for (long long base0 = gtid - lane; base0 < n4; base0 += UNI_UNR * nthreads) {
            float4 v[UNI_UNR];
            unsigned int m[UNI_UNR];
#pragma unroll
            for (int u = 0; u < UNI_UNR; ++u) {
                const long long i = base0 + lane + u * nthreads;
                v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                m[u] = 0u;
                if (i < n4) {
                    m[u] = P.mask ? __ldg(m4 + i) : 0x01010101u;
                    if (m[u]) v[u] = __ldcs(x4 + i);
                }
            }
#pragma unroll
            for (int u = 0; u < UNI_UNR; ++u) {
                if (__ballot_sync(0xffffffffu, m[u] != 0u) == 0u) continue;   // 128 unmasked samples: skipped whole
                add(v[u].x, (m[u] & 0xffu) != 0u);
                add(v[u].y, (m[u] & 0xff00u) != 0u);
                add(v[u].z, (m[u] & 0xff0000u) != 0u);
                add(v[u].w, (m[u] & 0xff000000u) != 0u);
            }
        }
        for (long long i0 = (n4 << 2) + gtid - lane; i0 < n; i0 += nthreads) {
            const long long i = i0 + lane;
            const bool use = i < n && (P.mask == nullptr || P.mask[i] != 0);
            add(use ? __ldg(xs + i) : 0.f, use);
        }
    }
    // the block's counts -> the series' u64 histograms
    __syncthreads();
    unsigned long long* hu = P.hu + (size_t)s * HS;
    for (int i = tid; i < R * 256; i += UNI_THREADS)
        if ((&h[0][0])[i]) atomicAdd(hu + i, (unsigned long long)(&h[0][0])[i]);
    if (P.pass == 0) {
        nan = __reduce_add_sync(0xffffffffu, nan);
        if (lane == 0) red[warp] = nan;
        __syncthreads();
        if (tid == 0) {
            unsigned int t = 0u;
            for (int w = 0; w < UNI_THREADS / 32; ++w) t += red[w];
            if (t) atomicAdd(hu + HS - 1, (unsigned long long)t);
        }
    }
    // the series' last block to finish writes the f64 image of its totals (the union so far: one unit after another)
    __threadfence();
    __syncthreads();
    if (tid == 0) last = atomicAdd(&P.ser[s].ticket, 1u) == gridDim.x - 1u;
    __syncthreads();
    if (!last) return;
    __threadfence();
    double* hf = P.hf + (size_t)s * HS;
    for (int i = tid; i < R * 256; i += UNI_THREADS) hf[i] = (double)__ldcg(hu + i);
    if (tid == 0) {
        if (P.pass == 0) hf[HS - 1] = (double)__ldcg(hu + HS - 1);
        P.ser[s].ticket = 0u;
    }
}

// One block per series, warp t = target t: reads the SUMMED histograms, picks every target's digit, then clears the
// histograms for the next pass.  Pass 0 also forms numpy's ranks from the union's sample count; the last pass writes
// the percentiles.
__global__ void __launch_bounds__(32 * SEL_MAXR) union_step_kernel(const UnionHead* hd, int Q, int pass, UnionSeries* ser, unsigned long long* hu, double* hf,
                                                                    double* out) {
    __shared__ unsigned int dead;
    const int s = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int T = 2 * Q, HS = union_hist_stride(Q);
    UnionSeries* sr = ser + s;
    double* hs = hf + (size_t)s * HS;
    if (tid == 0) dead = sr->dead;
    __syncthreads();
    if (pass == 0 && warp == 0) {                            // n = the union's masked non-NaN samples
        unsigned long long n = 0ull;
#pragma unroll
        for (int j = 0; j < 8; ++j) n += (unsigned long long)hs[lane * 8 + j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
        if (lane == 0) {
            if (n == 0ull || hs[HS - 1] != 0.0) {
                dead = 1u;
            } else {
                for (int j = 0; j < Q; ++j) {
                    long long r0, r1;
                    double gamma;
                    numpy_ranks((long long)n, hd->q[j], r0, r1, gamma);
                    sr->rank[2 * j] = (unsigned long long)r0;
                    sr->rank[2 * j + 1] = (unsigned long long)r1;
                    sr->gamma[j] = gamma;
                }
            }
        }
    }
    __syncthreads();
    if (dead == 0u && warp < T) {                            // lane l owns bins 8 l .. 8 l + 7
        const double* hb = hs + (pass == 0 ? 0 : warp * 256);
        unsigned long long c[8], local = 0ull;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            c[j] = (unsigned long long)hb[lane * 8 + j];
            local += c[j];
        }
        unsigned long long incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        unsigned long long excl = incl - local;
        const unsigned long long rk = sr->rank[warp];
        const unsigned int pre = pass == 0 ? 0u : sr->prefix[warp];
        const bool mine = rk >= excl && rk < excl + local;
        if (mine) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (rk >= excl && rk < excl + c[j]) {
                    sr->prefix[warp] = (pre << 8) | (unsigned int)(lane * 8 + j);
                    sr->rank[warp] = rk - excl;
                }
                excl += c[j];
            }
        }
        if (__ballot_sync(0xffffffffu, mine) == 0u && lane == 0) dead = 1u;   // the processes' calls did not match
    }
    __syncthreads();
    if (pass == 3 && tid < Q)
        out[(size_t)s * Q + tid] = dead ? __longlong_as_double(0x7ff8000000000000LL)
                                        : numpy_lerp(sr->prefix[2 * tid], sr->prefix[2 * tid + 1], sr->gamma[tid]);
    if (tid == 0) sr->dead = dead;
    for (int i = tid; i < HS; i += blockDim.x) {
        hs[i] = 0.0;
        hu[(size_t)s * HS + i] = 0ull;
    }
}

// out = (f32) clip((f64(x) - lo) / (hi - lo + 1e-12), 0, 1), series s = k * G + g   (color.py:33)
struct StretchParams {
    const float* x;
    long long xks, xgs;
    float* out;
    long long oks, ogs;
    const double* lohi;  // [S][2]
    long long n;
    int G, vec;
};

__global__ void __launch_bounds__(256) stretch_kernel(const StretchParams P) {
    const long long s = blockIdx.y;
    const long long k = s / P.G, g = s - k * P.G;
    const float* xs = P.x + k * P.xks + g * P.xgs;
    float* os = P.out + k * P.oks + g * P.ogs;
    const double lo = P.lohi[2 * s], den = P.lohi[2 * s + 1] - lo + 1e-12;
    auto f = [&](float v) {
        double r = ((double)v - lo) / den;
        r = r < 0.0 ? 0.0 : (r > 1.0 ? 1.0 : r);  // NaN survives, as np.clip
        return (float)r;
    };
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long n4 = P.vec ? (P.n >> 2) : 0;
    for (long long i = tid; i < n4; i += nthreads) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(xs) + i);
        __stcs(reinterpret_cast<float4*>(os) + i, make_float4(f(v.x), f(v.y), f(v.z), f(v.w)));
    }
    for (long long i = (n4 << 2) + tid; i < P.n; i += nthreads) os[i] = f(__ldg(xs + i));
}

// out = clip((f64(x) - lo) / (hi - lo + 1e-12), 0, 1) as float64, NaN outside the mask: robust_norm / robust_norm_rgb
// (color.py:6-23), whose results are float64 arrays
struct Stretch64Params {
    const float* x;
    long long xks, xgs;
    double* out;
    long long oks, ogs;
    const double* lohi;
    const uint8_t* mask;    // nullable: [G][n]
    long long n;
    int G;
};

__global__ void __launch_bounds__(256) stretch64_kernel(const Stretch64Params P) {
    const long long s = blockIdx.y;
    const long long k = s / P.G, g = s - k * P.G;
    const float* xs = P.x + k * P.xks + g * P.xgs;
    double* os = P.out + k * P.oks + g * P.ogs;
    const uint8_t* ms = P.mask ? P.mask + g * P.n : nullptr;
    const double lo = P.lohi[2 * s], den = P.lohi[2 * s + 1] - lo + 1e-12;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P.n; i += (long long)gridDim.x * blockDim.x) {
        double r = ((double)__ldg(xs + i) - lo) / den;
        r = r < 0.0 ? 0.0 : (r > 1.0 ? 1.0 : r);  // NaN survives, as np.clip
        if (ms && !ms[i]) r = __longlong_as_double(0x7ff8000000000000LL);
        os[i] = r;
    }
}

// out[i] = !isnan(x[i]) (& base[i]): the sample set of np.nanpercentile as a mask for the select kernels
__global__ void __launch_bounds__(256) notnan_mask_kernel(const float* __restrict__ x, const uint8_t* __restrict__ base,
                                                          long long n, uint8_t* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = __ldg(x + i);
        out[i] = (v == v && (base == nullptr || base[i])) ? 1 : 0;
    }
}

// ---- histogram matching (color.py:36-61): flags of the last element of every run of equal values in a sorted array
__global__ void __launch_bounds__(256) run_end_kernel(const float* __restrict__ v, long long n, uint8_t* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = (i == n - 1 || !(v[i] == v[i + 1])) ? 1 : 0;
}

// number of elements <= x in the ascending array v[0, n)
__device__ __forceinline__ long long count_le(const float* __restrict__ v, long long n, float x) {
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (v[mid] <= x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// One thread per pixel.  Masked pixels: q = (#source samples <= x) / ns  (the source CDF at x, color.py:44-47), then
// np.interp(q, r_quant, r_values) (:49) with r_quant[j] = (end[j] + 1) / nr the reference CDF at its j-th distinct value
// r_values[j] = ref_sorted[end[j]] — numpy's arithmetic: one division per quantile, slope * (x - xp[j]) + fp[j] without
// contraction — cast to float32; every pixel is then clipped to [0, 1] (:60).
__global__ void __launch_bounds__(256) hist_match_kernel(const float* __restrict__ src, const uint8_t* __restrict__ mask,
                                                         long long n, const float* __restrict__ src_sorted, long long ns,
                                                         const float* __restrict__ ref_sorted, long long nr,
                                                         const int* __restrict__ end, long long nu, float* __restrict__ out) {
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        float x = src[p];
        if (mask[p]) {
            const double q = (double)count_le(src_sorted, ns, x) / (double)ns;
            const double x_first = (double)(end[0] + 1) / (double)nr, x_last = (double)(end[nu - 1] + 1) / (double)nr;
            double r;
            if (q > x_last) {
                r = (double)ref_sorted[end[nu - 1]];
            } else if (q < x_first) {
                r = (double)ref_sorted[end[0]];
            } else {
                long long lo = 0, hi = nu;                       // largest j with r_quant[j] <= q
                while (hi - lo > 1) {
                    const long long mid = (lo + hi) >> 1;
                    if ((double)(end[mid] + 1) / (double)nr <= q) lo = mid;
                    else hi = mid;
                }
                const double xj = (double)(end[lo] + 1) / (double)nr, fj = (double)ref_sorted[end[lo]];
                if (lo == nu - 1 || xj == q) {
                    r = fj;
                } else {
                    const double xk = (double)(end[lo + 1] + 1) / (double)nr, fk = (double)ref_sorted[end[lo + 1]];
                    const double slope = __ddiv_rn(__dsub_rn(fk, fj), __dsub_rn(xk, xj));
                    r = __dadd_rn(__dmul_rn(slope, __dsub_rn(q, xj)), fj);
                }
            }
            x = (float)r;
        }
        out[p] = x < 0.f ? 0.f : (x > 1.f ? 1.f : x);             // NaN survives, as np.clip
    }
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

int run_ends_impl(const float* sorted, long long n, uint8_t* flags, cudaStream_t stream) {
    HSR_REQUIRE(sorted && flags, HSR_EINVAL, "null sorted / flags pointer");
    HSR_REQUIRE(n >= 0, HSR_EINVAL, "negative n");
    if (n == 0) return HSR_OK;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)device_sm_count() * 8;
    run_end_kernel<<<(unsigned int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(sorted, n, flags);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int hist_match_impl(const float* src, const uint8_t* mask, long long n, const float* src_sorted, long long ns,
                    const float* ref_sorted, long long nr, const int* ref_run_ends, long long nu, float* out,
                    cudaStream_t stream) {
    HSR_REQUIRE(src && mask && src_sorted && ref_sorted && ref_run_ends && out, HSR_EINVAL, "null pointer");
    HSR_REQUIRE(n >= 0 && ns >= 1 && nr >= 1 && nu >= 1 && nu <= nr && nr < 2147483647LL, HSR_ERANGE,
                "need n >= 0, ns >= 1, 1 <= nu <= nr < 2^31 (got %lld, %lld, %lld, %lld)", n, ns, nu, nr);
    if (n == 0) return HSR_OK;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)device_sm_count() * 8;
    hist_match_kernel<<<(unsigned int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(src, mask, n, src_sorted, ns, ref_sorted,
                                                                                     nr, ref_run_ends, nu, out);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int stretch64_impl(const float* x, long long xks, long long xgs, const double* lohi, const uint8_t* mask, long long n,
                   int K, int G, double* out, long long oks, long long ogs, cudaStream_t stream) {
    HSR_REQUIRE(x && lohi && out, HSR_EINVAL, "null x / lohi / out pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && G >= 1 && (long long)K * G <= 65535, HSR_ERANGE,
                "bad n = %lld, K = %d or G = %d (K * G <= 65535)", n, K, G);
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(x) & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0, HSR_EALIGN,
                "x not 4-byte / out not 8-byte aligned");
    if (n == 0) return HSR_OK;
    Stretch64Params P{};
    P.x = x, P.xks = xks, P.xgs = xgs, P.out = out, P.oks = oks, P.ogs = ogs, P.lohi = lohi, P.mask = mask, P.n = n, P.G = G;
    const long long S = (long long)K * G;
    long long per = (n + 256 * 4 - 1) / (256 * 4);
    long long cap = (long long)device_sm_count() * 6 / S;
    if (cap < 1) cap = 1;
    dim3 grid((unsigned int)(per < cap ? per : cap), (unsigned int)S);
    stretch64_kernel<<<grid, 256, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int notnan_mask_impl(const float* x, const uint8_t* base, long long n, uint8_t* out, cudaStream_t stream) {
    HSR_REQUIRE(x && out, HSR_EINVAL, "null x / out pointer");
    HSR_REQUIRE(n >= 0, HSR_EINVAL, "negative n");
    if (n == 0) return HSR_OK;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)device_sm_count() * 8;
    notnan_mask_kernel<<<(unsigned int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(x, base, n, out);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

// candidates kept per bracket: ~1 % of a series falls inside a bracket; small series need proportionally less
static unsigned int sel_capacity(long long n) {
    long long c = n / 16;
    if (c < 4096) c = 4096;
    if (c > SEL_CAP) c = SEL_CAP;
    if (c > n && n > 0) c = n;                        // a series never has more candidates than samples
    return (unsigned int)c;
}

size_t percentiles_workspace(long long n, int K, int G, int nsets) {
    if (K < 1 || G < 1 || n < 0 || nsets < 1 || nsets > 2) return 0;
    const size_t S = (size_t)K * (size_t)G * (size_t)nsets;
    return align_up(S * sizeof(SelSeries), 256) + S * SEL_QMAX * (size_t)sel_capacity(n) * sizeof(unsigned int);
}

// x2 (nullable): a second plane set of the same shape (the reference image of the stretch, poly_regression.py:126-127)
// handled by the same three launches; out2 receives its percentiles.
int masked_percentiles_impl(const float* x, long long xks, long long xgs, const float* x2, long long x2ks, long long x2gs,
                            const uint8_t* mask, long long n, int K, int G, const double* q, int Q, void* workspace,
                            double* out, double* out2, cudaStream_t stream) {
    HSR_REQUIRE(x && q && workspace && out, HSR_EINVAL, "null x / q / workspace / out pointer");
    HSR_REQUIRE((x2 == nullptr) == (out2 == nullptr), HSR_EINVAL, "x2 and out2 must be given together");
    // n < 2^32: the candidate counts (SelSeries::ncand, nc) and the fallback's histogram bins are 32-bit; a wrapped ncand
    // could pass as <= cap and send the finish kernel to a candidate list it never filled
    HSR_REQUIRE(n >= 0 && n < (1LL << 32) && K >= 1 && G >= 1 && (long long)K * G <= 32767, HSR_ERANGE,
                "bad n = %lld (< 2^32), K = %d or G = %d (K * G <= 32767)", n, K, G);
    HSR_REQUIRE(Q >= 1 && Q <= SEL_QMAX, HSR_ERANGE, "Q = %d outside [1, %d]", Q, SEL_QMAX);
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(x2)) & 3) == 0, HSR_EALIGN,
                "x not 4-byte aligned");
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, HSR_EALIGN, "workspace not 256-byte aligned");
    const long long S1 = (long long)K * G;
    SelParams P{};
    P.nsets = x2 ? 2 : 1;
    const long long S = S1 * P.nsets;
    P.x[0] = x, P.xks[0] = xks, P.xgs[0] = xgs, P.out[0] = out;
    P.x[1] = x2, P.xks[1] = x2ks, P.xgs[1] = x2gs, P.out[1] = out2;
    P.S1 = S1, P.mask = mask, P.n = n, P.G = G, P.Q = Q, P.q = q;
    P.cap = sel_capacity(n);
    P.st = reinterpret_cast<SelSeries*>(workspace);
    P.cand = reinterpret_cast<unsigned int*>(reinterpret_cast<unsigned char*>(workspace) +
                                             align_up((size_t)S * sizeof(SelSeries), 256));
    const uintptr_t a4 = reinterpret_cast<uintptr_t>(mask) | (uintptr_t)(G > 1 ? n : 0);
    for (int i = 0; i < P.nsets; ++i) {
        const long long s_or = (K > 1 ? P.xks[i] : 0) | (G > 1 ? P.xgs[i] : 0);
        const uintptr_t a16 = reinterpret_cast<uintptr_t>(P.x[i]) | (uintptr_t)(s_or * 4);
        P.vec[i] = ((a16 & 15) == 0 && (a4 & 3) == 0) ? 1 : 0;
    }
    select_sample_kernel<<<(unsigned int)S, SEL_BT, 0, stream>>>(P);
    long long per = (n + (long long)SEL_THREADS * 16 - 1) / ((long long)SEL_THREADS * 16);
    if (per < 1) per = 1;
    long long cap = (long long)device_sm_count() * 8 / S;
    if (cap < 1) cap = 1;
    dim3 grid((unsigned int)(per < cap ? per : cap), (unsigned int)S);
    select_collect_kernel<<<grid, SEL_THREADS, 0, stream>>>(P);
    const size_t fsmem = (size_t)P.cap * sizeof(unsigned int);
    static int smem_set[HSR_MAX_DEVICES];
    HSR_CUDA(ensure_dynamic_smem(select_finish_kernel, (int)(SEL_CAP * sizeof(unsigned int)), smem_set));
    select_finish_kernel<<<dim3((unsigned int)S, (unsigned int)Q), SEL_BT, fsmem, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

// union select state: UnionHead | UnionSeries[S] | u64 histograms [S][HS], each part 256-byte aligned
static size_t union_head_bytes() { return align_up(sizeof(UnionHead), 256); }
static size_t union_series_bytes(int S) { return align_up((size_t)S * sizeof(UnionSeries), 256); }

static bool union_args_ok(int Q, int S) { return Q >= 1 && Q <= SEL_QMAX && S >= 1 && S <= 65535; }

size_t union_state_bytes(int Q, int S) {
    if (!union_args_ok(Q, S)) return 0;
    return union_head_bytes() + union_series_bytes(S) + (size_t)S * union_hist_stride(Q) * sizeof(unsigned long long);
}

long long union_hist_doubles(int Q, int S) {
    return union_args_ok(Q, S) ? (long long)S * union_hist_stride(Q) : 0;
}

struct UnionState {
    UnionHead* hd;
    UnionSeries* ser;
    unsigned long long* hu;
};

static UnionState union_state(void* state, int S) {
    unsigned char* b = reinterpret_cast<unsigned char*>(state);
    return {reinterpret_cast<UnionHead*>(b), reinterpret_cast<UnionSeries*>(b + union_head_bytes()),
            reinterpret_cast<unsigned long long*>(b + union_head_bytes() + union_series_bytes(S))};
}

int union_begin_impl(const double* q, int Q, int S, void* state, double* hist, cudaStream_t stream) {
    HSR_REQUIRE(q && state && hist, HSR_EINVAL, "null q / state / hist pointer");
    HSR_REQUIRE(union_args_ok(Q, S), HSR_ERANGE, "Q = %d outside [1, %d] or S = %d outside [1, 65535]", Q, SEL_QMAX, S);
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(state) & 255) == 0 && (reinterpret_cast<uintptr_t>(hist) & 7) == 0,
                HSR_EALIGN, "state not 256-byte / hist not 8-byte aligned");
    HSR_CUDA(cudaMemsetAsync(state, 0, union_state_bytes(Q, S), stream));
    HSR_CUDA(cudaMemsetAsync(hist, 0, (size_t)union_hist_doubles(Q, S) * sizeof(double), stream));
    HSR_CUDA(cudaMemcpyAsync(union_state(state, S).hd->q, q, (size_t)Q * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    return HSR_OK;
}

int union_count_impl(const float* x, long long xks, const float* y, long long yks, const uint8_t* mask, long long n,
                     int K, int Q, int pass, void* state, double* hist, cudaStream_t stream) {
    HSR_REQUIRE(state && hist, HSR_EINVAL, "null state / hist pointer");
    const long long S = (long long)K * (y ? 2 : 1);
    // n < 2^32 per unit: the per-block counters are 32-bit (the union's totals are 64-bit)
    HSR_REQUIRE(n >= 0 && n < (1LL << 32) && K >= 1 && S <= 65535 && union_args_ok(Q, (int)S), HSR_ERANGE,
                "bad n = %lld (< 2^32), K = %d (K * sets <= 65535) or Q = %d", n, K, Q);
    HSR_REQUIRE(pass >= 0 && pass <= 3, HSR_ERANGE, "pass = %d outside [0, 3]", pass);
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 3) == 0, HSR_EALIGN,
                "x / y not 4-byte aligned");
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(state) & 255) == 0, HSR_EALIGN, "state not 256-byte aligned");
    if (n == 0) return HSR_OK;                       // an empty unit adds nothing (its planes may have no storage)
    HSR_REQUIRE(x, HSR_EINVAL, "null x pointer");
    const UnionState us = union_state(state, (int)S);
    UnionCountParams P{};
    P.x[0] = x, P.xks[0] = xks, P.x[1] = y, P.xks[1] = yks;
    P.mask = mask, P.n = n, P.K = K, P.S = (int)S, P.Q = Q, P.pass = pass;
    P.ser = us.ser, P.hu = us.hu, P.hf = hist;
    for (int i = 0; i < (y ? 2 : 1); ++i) {
        const uintptr_t a16 = reinterpret_cast<uintptr_t>(P.x[i]) | (uintptr_t)((K > 1 ? P.xks[i] : 0) * 4);
        P.vec[i] = ((a16 & 15) == 0 && (reinterpret_cast<uintptr_t>(mask) & 3) == 0) ? 1 : 0;
    }
    long long per = (n + (long long)UNI_THREADS * 4 * UNI_UNR - 1) / ((long long)UNI_THREADS * 4 * UNI_UNR);
    long long cap = (long long)device_sm_count() * 8 / S;
    if (cap < 1) cap = 1;
    const dim3 grid((unsigned int)(per < cap ? per : cap), (unsigned int)S);
    if (pass == 0) union_count_kernel<1><<<grid, UNI_THREADS, 0, stream>>>(P);
    else if (Q == 1) union_count_kernel<2><<<grid, UNI_THREADS, 0, stream>>>(P);
    else union_count_kernel<2 * SEL_QMAX><<<grid, UNI_THREADS, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int union_step_impl(int Q, int S, int pass, void* state, double* hist, double* out, int* more, cudaStream_t stream) {
    HSR_REQUIRE(state && hist, HSR_EINVAL, "null state / hist pointer");
    HSR_REQUIRE(union_args_ok(Q, S), HSR_ERANGE, "Q = %d outside [1, %d] or S = %d outside [1, 65535]", Q, SEL_QMAX, S);
    HSR_REQUIRE(pass >= 0 && pass <= 3, HSR_ERANGE, "pass = %d outside [0, 3]", pass);
    HSR_REQUIRE(pass < 3 || out, HSR_EINVAL, "null out pointer on the last pass");
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(state) & 255) == 0, HSR_EALIGN, "state not 256-byte aligned");
    const UnionState us = union_state(state, S);
    union_step_kernel<<<(unsigned int)S, 64 * Q, 0, stream>>>(us.hd, Q, pass, us.ser, us.hu, hist, out);
    HSR_CUDA(cudaGetLastError());
    if (more) *more = pass < 3 ? 1 : 0;
    return HSR_OK;
}

int stretch_impl(const float* x, long long xks, long long xgs, const double* lohi, long long n, int K, int G,
                 float* out, long long oks, long long ogs, cudaStream_t stream) {
    HSR_REQUIRE(x && lohi && out, HSR_EINVAL, "null x / lohi / out pointer");
    HSR_REQUIRE(n >= 0 && K >= 1 && G >= 1 && (long long)K * G <= 65535, HSR_ERANGE,
                "bad n = %lld, K = %d or G = %d (K * G <= 65535)", n, K, G);
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 3) == 0, HSR_EALIGN,
                "x / out not 4-byte aligned");
    if (n == 0) return HSR_OK;
    StretchParams P{};
    P.x = x, P.xks = xks, P.xgs = xgs, P.out = out, P.oks = oks, P.ogs = ogs, P.lohi = lohi, P.n = n, P.G = G;
    const long long s_or = (K > 1 ? (xks | oks) : 0) | (G > 1 ? (xgs | ogs) : 0);
    P.vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | (uintptr_t)(s_or * 4)) & 15) == 0;
    const long long S = (long long)K * G;
    long long per = (n + 256 * 8 - 1) / (256 * 8);
    long long cap = (long long)device_sm_count() * 6 / S;
    if (cap < 1) cap = 1;
    dim3 grid((unsigned int)(per < cap ? per : cap), (unsigned int)S);
    stretch_kernel<<<grid, 256, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

}  // namespace hsr
