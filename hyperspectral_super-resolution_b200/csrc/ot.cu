// ot.cu — the optimal-transport target stage of fit_ot_poly_rgb (SURVEY section 8 row a8):
// s2_emit/poly_regression.py:31-60
//     X_all = src[mask] rows with every channel finite (row-major order), likewise Y_all          :33-36
//     X, Y  = rng.choice samples of them (the index draw stays on the host: numpy's generator)     :46-47
//     M = ot.dist(X, Y, "sqeuclidean");  P = ot.sinkhorn(a, b, M, reg, numItermax, stopThr)         :52-53
//     Ybar = (P @ Y) / (P.sum(1) + 1e-32)                                                         :55-56
//     coeffs[c] = np.polyfit(X[:, c], Ybar[:, c], deg)                                             :58-60
// POT (import name `ot`) is a third-party dependency that is neither vendored nor pinned by the reference; the
// kernels follow its published algorithms: ot.dist -> euclidean_distances(squared=True)
// (|x|^2 + |y|^2 - 2 x.y, clamped at 0) and ot.sinkhorn -> sinkhorn_knopp (K = exp(M / -reg), u = v = 1/n,
// v = b / K^T u, u = 1 / (diag(1/a) K) v, marginal error every 10th iteration, roll back and stop on
// 0 / NaN / Inf).  Everything is fp64.
//
// The kernel matrix K (ns x nt fp64, 200 MB at the reference's 5000 x 5000) is built once and streamed twice
// per iteration: a column pass (K^T u, rows split into chunks, partials summed in a fixed order) and a row pass
// (one warp per row).  All numItermax iterations are enqueued up front; convergence and the numerical-error
// roll-back are device-side flags that turn the remaining launches into no-ops, so there is no host round trip.
// The every-10th-iteration marginal check needs K^T u_new, which IS the next iteration's column pass, so it
// costs no extra sweep.
#include <stdlib.h>

#include "hsr_common.cuh"

namespace hsr {

namespace {

constexpr int OT_MAXC = 4;       // channels per sample (RGB = 3)
constexpr int COL_THREADS = 128;
constexpr int OT_PARTS_MAX = 160;   // column-pass partial rows: <= 32 chunks, or one per SM in the fused kernel

struct OtState {
    int done;          // 1: stop iterating (converged or numerical error)
    int errflag;       // set by an iteration that produced 0 / NaN / Inf: roll back to the previous u, v
    int final_it;      // u, v of this iteration index are the result (buffer parity = final_it & 1)
    int numerical;     // stopped because of a numerical error
    double err;        // last marginal violation that was evaluated
    int err_it;
    unsigned int ticket;  // blocks of the current v-update that have finished (the last one decides)
    int it;               // iteration counter of the device-side loop (CUDA-graph WHILE node)
};

// ---------------------------------------------------------------------------------- compaction
// flags[i] = mask[i] && all_c isfinite(img[i, c]); order-preserving compaction of the row indices.
__global__ void __launch_bounds__(256) compact_count_kernel(const float* __restrict__ img, const uint8_t* __restrict__ mask,
                                                            long long n, int C, int rows_per_block,
                                                            unsigned int* __restrict__ block_count) {
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    unsigned int c = 0;
    for (long long i = r0 + threadIdx.x; i < r0 + rows_per_block && i < n; i += 256) {
        bool f = mask == nullptr || mask[i] != 0;
        for (int k = 0; k < C; ++k) f = f && finite_f32(__ldg(img + i * C + k));
        c += f ? 1u : 0u;
    }
    __shared__ unsigned int red[8];
    c = (unsigned int)warp_sum((int)c);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
        for (int w = 0; w < 8; ++w) t += red[w];
        block_count[blockIdx.x] = t;
    }
}

__global__ void compact_scan_kernel(const unsigned int* __restrict__ block_count, int nblocks,
                                    long long* __restrict__ block_base, long long* __restrict__ total) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        long long run = 0;
        for (int b = 0; b < nblocks; ++b) {
            block_base[b] = run;
            run += block_count[b];
        }
        *total = run;
    }
}

__global__ void __launch_bounds__(256) compact_scatter_kernel(const float* __restrict__ img, const uint8_t* __restrict__ mask,
                                                              long long n, int C, int rows_per_block,
                                                              const long long* __restrict__ block_base,
                                                              int* __restrict__ idx) {
    __shared__ unsigned int wcount[8];
    __shared__ long long base_s;
    const long long r0 = (long long)blockIdx.x * rows_per_block;
    if (threadIdx.x == 0) base_s = block_base[blockIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long long s0 = r0; s0 < r0 + rows_per_block && s0 < n; s0 += 256) {
        const long long i = s0 + threadIdx.x;
        bool f = i < n && i < r0 + rows_per_block && (mask == nullptr || mask[i] != 0);
        if (f)
            for (int k = 0; k < C; ++k) f = f && finite_f32(__ldg(img + i * C + k));
        const unsigned int b = __ballot_sync(0xffffffffu, f);
        if (lane == 0) wcount[warp] = __popc(b);
        __syncthreads();
        long long off = base_s;
        for (int w = 0; w < warp; ++w) off += wcount[w];
        if (f) idx[off + __popc(b & ((1u << lane) - 1u))] = (int)i;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int t = 0;
            for (int w = 0; w < 8; ++w) t += wcount[w];
            base_s += t;
        }
        __syncthreads();
    }
}

// out[r, c] = (f64) img[idx[sel[r]], c]     (X = X_all[rng.choice(...)], :46-47, after .astype(float64) :33)
__global__ void gather_rows_kernel(const float* __restrict__ img, const int* __restrict__ idx,
                                   const long long* __restrict__ sel, long long ns, int C, double* __restrict__ out) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= ns * C) return;
    const long long r = t / C;
    const int c = (int)(t - r * C);
    out[t] = (double)__ldg(img + (long long)idx[sel[r]] * C + c);
}

// ---------------------------------------------------------------------------------- Sinkhorn
// K[i, j] = exp(max(|x_i|^2 + |y_j|^2 - 2 x_i.y_j, 0) / -reg)      (ot.dist + the first line of sinkhorn_knopp)
__global__ void __launch_bounds__(256) ot_kernel_matrix(const double* __restrict__ X, const double* __restrict__ Y,
                                                        int ns, int nt, int C, double reg, double* __restrict__ K) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    const int i0 = blockIdx.y * 16;
    if (j >= nt) return;
    double y[OT_MAXC], b2 = 0.0;
    for (int c = 0; c < C; ++c) {
        y[c] = Y[(long long)j * C + c];
        b2 = fma(y[c], y[c], b2);
    }
    for (int i = i0; i < i0 + 16 && i < ns; ++i) {
        double a2 = 0.0, d = 0.0;
        for (int c = 0; c < C; ++c) {
            const double x = X[(long long)i * C + c];
            a2 = fma(x, x, a2);
            d = fma(x, y[c], d);
        }
        double m = (-2.0 * d + a2) + b2;
        m = m > 0.0 ? m : 0.0;
        K[(long long)i * nt + j] = exp(m / (-reg));
    }
}

__global__ void ot_init_kernel(double* __restrict__ u, double* __restrict__ v, int ns, int nt, OtState* st) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ns) u[t] = 1.0 / ns;   // buffer 0 = iteration 0
    if (t < nt) v[t] = 1.0 / nt;
    if (t == 0) {
        st->done = 0;
        st->errflag = 0;
        st->final_it = 0;
        st->numerical = 0;
        st->err = 1.0;
        st->err_it = -1;
        st->ticket = 0u;
        st->it = 0;
    }
}

// Column pass of iteration `it`: partial[chunk, j] = sum_{i in chunk} K[i, j] * u_it[i]
__global__ void __launch_bounds__(COL_THREADS) ot_colpass_kernel(const double* __restrict__ K, const double* __restrict__ ubuf,
                                                                 int ns, int nt, int it, int rows_per_chunk,
                                                                 double* __restrict__ partial, const OtState* st) {
    if (st->done || st->errflag) return;
    extern __shared__ double us[];
    const double* u = ubuf + (long long)(it & 1) * ns;
    const int r0 = blockIdx.y * rows_per_chunk;
    int r1 = r0 + rows_per_chunk;
    if (r1 > ns) r1 = ns;
    for (int i = r0 + threadIdx.x; i < r1; i += COL_THREADS) us[i - r0] = u[i];
    __syncthreads();
    const int j = blockIdx.x * COL_THREADS + threadIdx.x;
    if (j >= nt) return;
    const double* kp = K + (long long)r0 * nt + j;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int i = 0;
    const int nr = r1 - r0;
    for (; i + 3 < nr; i += 4) {
        const double k0 = kp[(long long)i * nt], k1 = kp[(long long)(i + 1) * nt];
        const double k2 = kp[(long long)(i + 2) * nt], k3 = kp[(long long)(i + 3) * nt];
        s0 = fma(k0, us[i], s0);
        s1 = fma(k1, us[i + 1], s1);
        s2 = fma(k2, us[i + 2], s2);
        s3 = fma(k3, us[i + 3], s3);
    }
    for (; i < nr; ++i) s0 = fma(kp[(long long)i * nt], us[i], s0);
    partial[(long long)blockIdx.y * nt + j] = (s0 + s1) + (s2 + s3);
}

// KtU = sum of the column-pass partials (fixed order), 256 columns per block.  If the previous iteration was a
// multiple of 10, its marginal check err = || v * KtU - b ||_2 happens here (u, v are the updated ones; KtU is
// exactly the einsum('i,ij,j->j') column sums).  v_{it+1} = b / KtU is written speculatively into the other
// buffer; the LAST block to finish (ticket) adds the per-block error terms in a fixed order and decides:
// converged -> done with (u_it, v_it); zeros / NaN / Inf -> errflag (rolled back by the next launch).
constexpr int VUP_THREADS = 256;
constexpr int VUP_COLS = 32;
constexpr int VUP_SLICES = VUP_THREADS / VUP_COLS;

__global__ void __launch_bounds__(VUP_THREADS) ot_vupdate_kernel(const double* __restrict__ partial, int nparts, int ns, int nt,
                                                                 int it_arg, double bval, double stop_thr,
                                                                 double* __restrict__ vbuf, double* __restrict__ e2part,
                                                                 int* __restrict__ badpart, OtState* st) {
    __shared__ double red[VUP_THREADS / 32];
    __shared__ int bad_s;
    if (st->done) return;
    const int it = it_arg >= 0 ? it_arg : st->it;  // < 0: inside the device-side loop, the counter lives in *st
    if (st->errflag) {  // the previous iteration broke down: its predecessor's u, v are the result
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            st->done = 1;
            st->numerical = 1;
            st->final_it = it - 1;
        }
        return;
    }
    const double* v = vbuf + (long long)(it & 1) * nt;
    double* vn = vbuf + (long long)((it + 1) & 1) * nt;
    const bool check = it > 0 && ((it - 1) % 10) == 0;
    if (threadIdx.x == 0) bad_s = 0;
    __syncthreads();
    // 32 columns per block; the 8 threads of a column each sum every 8th partial row (independent loads in
    // flight), then the 8 slice sums are added in a fixed order
    __shared__ double slice[VUP_SLICES][VUP_COLS];
    const int cl = threadIdx.x & (VUP_COLS - 1), sl = threadIdx.x / VUP_COLS;
    const int j = blockIdx.x * VUP_COLS + cl;
    double ps = 0.0;
    if (j < nt) {
        double p0 = 0.0, p1 = 0.0, p2 = 0.0, p3 = 0.0;
        int c = sl;
        for (; c + 3 * VUP_SLICES < nparts; c += 4 * VUP_SLICES) {
            p0 += partial[(long long)c * nt + j];
            p1 += partial[(long long)(c + VUP_SLICES) * nt + j];
            p2 += partial[(long long)(c + 2 * VUP_SLICES) * nt + j];
            p3 += partial[(long long)(c + 3 * VUP_SLICES) * nt + j];
        }
        for (; c < nparts; c += VUP_SLICES) p0 += partial[(long long)c * nt + j];
        ps = (p0 + p1) + (p2 + p3);
    }
    slice[sl][cl] = ps;
    __syncthreads();
    double e2 = 0.0;
    if (sl == 0 && j < nt) {
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < VUP_SLICES; ++q) s += slice[q][cl];
        if (check) {
            const double d = v[j] * s - bval;
            e2 = d * d;
        }
        const double nv = bval / s;
        vn[j] = nv;
        if (s == 0.0 || isnan(nv) || isinf(nv)) bad_s = 1;
    }
    e2 = warp_sum(e2);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = e2;
    __syncthreads();
    __shared__ int last_s;
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < VUP_THREADS / 32; ++w) t += red[w];
        e2part[blockIdx.x] = t;
        badpart[blockIdx.x] = bad_s;
        __threadfence();
        last_s = (atomicAdd(&st->ticket, 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!last_s) return;
    // last block: every block's partial is visible; add them in a fixed order, in parallel
    __threadfence();
    double tot = 0.0;
    int bad = 0;
    for (unsigned int b = threadIdx.x; b < gridDim.x; b += VUP_THREADS) {
        tot += __ldcg(e2part + b);
        bad |= __ldcg(badpart + b);
    }
    tot = warp_sum(tot);
    bad = __any_sync(0xffffffffu, bad) ? 1 : 0;
    __shared__ int badw[VUP_THREADS / 32];
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = tot;
        badw[threadIdx.x >> 5] = bad;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        tot = 0.0;
        bad = 0;
        for (int w = 0; w < VUP_THREADS / 32; ++w) {
            tot += red[w];
            bad |= badw[w];
        }
        st->ticket = 0u;
        bool stop = false;
        if (check) {
            const double err = sqrt(tot);
            st->err = err;
            st->err_it = it - 1;
            stop = err < stop_thr;
        }
        if (stop) {
            st->done = 1;
            st->final_it = it;
        } else {
            if (bad) st->errflag = 1;
            st->final_it = it + 1;  // provisional: stands unless this iteration turns out bad
        }
    }
}

// Row pass: u_{it+1}[i] = 1 / sum_j ((1/a) * K[i, j]) * v_{it+1}[j]; one warp per row.
__global__ void __launch_bounds__(256) ot_rowpass_kernel(const double* __restrict__ K, const double* __restrict__ vbuf,
                                                         int ns, int nt, int it, double inv_a, double* __restrict__ ubuf,
                                                         OtState* st) {
    if (st->done || st->errflag) return;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= ns) return;
    const double* v = vbuf + (long long)((it + 1) & 1) * nt;
    const double* kr = K + (long long)row * nt;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int j = lane;
    for (; j + 96 < nt; j += 128) {
        const double k0 = kr[j], k1 = kr[j + 32], k2 = kr[j + 64], k3 = kr[j + 96];
        s0 = fma(inv_a * k0, v[j], s0);
        s1 = fma(inv_a * k1, v[j + 32], s1);
        s2 = fma(inv_a * k2, v[j + 64], s2);
        s3 = fma(inv_a * k3, v[j + 96], s3);
    }
    for (; j < nt; j += 32) s0 = fma(inv_a * kr[j], v[j], s0);
    const double s = warp_sum((s0 + s1) + (s2 + s3));
    if (lane == 0) {
        const double nu = 1.0 / s;
        ubuf[(long long)((it + 1) & 1) * ns + row] = nu;
        if (isnan(nu) || isinf(nu)) atomicOr(&st->errflag, 1);
    }
}

// Fused row pass of iteration `it` + column pass of iteration `it + 1`: both sweep the same rows of K, so K is
// read from HBM ONCE per iteration.  Persistent CTAs (one per SM); each takes whole rows, staged in shared memory
// by 1-D bulk copies (TMA) through a four-stage ring (three rows in flight while one is consumed).  Thread t owns
// columns j = t, t + 256, ...: it keeps v_{it+1}[j] and its column accumulators in registers for the whole kernel,
// reads its K[i, j] of the staged row ONCE, contributes to the row sum (u_{it+1}[i] = 1 / sum_j ((1/a) K[i, j]) v[j],
// block-reduced in a fixed order), then adds u_i K[i, j] to its accumulators.  One partial row of column sums per
// CTA goes to the v-update kernel.
constexpr int FUSE_THREADS = 256;
constexpr int FUSE_NST = 4;      // ring stages (rows)
constexpr int FUSE_NCMAX = 24;   // columns per thread: nt <= 24 * 256

__global__ void __launch_bounds__(FUSE_THREADS, 1) ot_fused_kernel(const double* __restrict__ K, const double* __restrict__ vbuf,
                                                                   double* __restrict__ ubuf, int ns, int nt, int it_arg,
                                                                   double inv_a, double* __restrict__ partial, OtState* st) {
    if (st->done || st->errflag) return;
    const int it = it_arg >= 0 ? it_arg : st->it;
    extern __shared__ __align__(128) unsigned char fsm[];
    uint64_t* full = reinterpret_cast<uint64_t*>(fsm);                       // [FUSE_NST]
    double* rs = reinterpret_cast<double*>(fsm + 64);                        // [2][8] warp sums, double-buffered
    double* stages = reinterpret_cast<double*>(fsm + 256);                   // [FUSE_NST][nt]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* v = vbuf + (long long)((it + 1) & 1) * nt;
    double* un = ubuf + (long long)((it + 1) & 1) * ns;
    const int mine = ((int)blockIdx.x < ns) ? (ns - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;  // my rows
    const unsigned int row_bytes = (unsigned int)nt * 8u;

    if (tid == 0) {
        for (int s = 0; s < FUSE_NST; ++s) mbar_init(&full[s], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](int idx) {  // thread 0 only: stage my idx-th row
        const int s = idx % FUSE_NST;
        const long long row = blockIdx.x + (long long)idx * gridDim.x;
        mbar_arrive_expect_tx(&full[s], row_bytes);
        bulk_g2s(stages + (long long)s * nt, K + row * nt, row_bytes, &full[s]);
    };
    if (tid == 0)
        for (int idx = 0; idx < FUSE_NST && idx < mine; ++idx) issue(idx);

    double vreg[FUSE_NCMAX], colacc[FUSE_NCMAX];
#pragma unroll
    for (int m = 0; m < FUSE_NCMAX; ++m) {
        const int j = tid + m * FUSE_THREADS;
        vreg[m] = j < nt ? v[j] : 0.0;
        colacc[m] = 0.0;
    }
    int bad = 0;
    for (int idx = 0; idx < mine; ++idx) {
        const int s = idx % FUSE_NST;
        const double* kst = stages + (long long)s * nt;
        mbar_wait(&full[s], (unsigned int)(idx / FUSE_NST) & 1u);
        double kreg[FUSE_NCMAX];
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int m = 0; m < FUSE_NCMAX; m += 2) {
            const int j0 = tid + m * FUSE_THREADS, j1 = j0 + FUSE_THREADS;
            kreg[m] = j0 < nt ? kst[j0] : 0.0;
            kreg[m + 1] = j1 < nt ? kst[j1] : 0.0;
            a0 = fma(inv_a * kreg[m], vreg[m], a0);
            a1 = fma(inv_a * kreg[m + 1], vreg[m + 1], a1);
        }
        const double t = warp_sum(a0 + a1);
        double* rsb = rs + (idx & 1) * 8;
        if (lane == 0) rsb[warp] = t;
        __syncthreads();  // every thread holds its part of the row in registers: the stage is free again
        if (tid == 0 && idx + FUSE_NST < mine) issue(idx + FUSE_NST);
        double sum = 0.0;
#pragma unroll
        for (int w = 0; w < FUSE_THREADS / 32; ++w) sum += rsb[w];
        const double ui = 1.0 / sum;
        if (tid == 0) {
            un[blockIdx.x + (long long)idx * gridDim.x] = ui;
            if (isnan(ui) || isinf(ui)) bad = 1;
        }
#pragma unroll
        for (int m = 0; m < FUSE_NCMAX; ++m) colacc[m] = fma(kreg[m], ui, colacc[m]);
    }
    if (bad) atomicOr(&st->errflag, 1);
#pragma unroll
    for (int m = 0; m < FUSE_NCMAX; ++m) {
        const int j = tid + m * FUSE_THREADS;
        if (j < nt) partial[(long long)blockIdx.x * nt + j] = colacc[m];
    }
}

// Tail of one iteration of the device-side loop: advance the counter and tell the WHILE node whether to go on.
__global__ void ot_step_kernel(OtState* st, cudaGraphConditionalHandle handle, int num_iter_max) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const int it = st->it + 1;
        st->it = it;
        cudaGraphSetConditional(handle, (!st->done && it < num_iter_max) ? 1u : 0u);
    }
}

// After the last iteration: an error raised by its row pass still rolls back.
__global__ void ot_finish_kernel(int num_iter, OtState* st) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && !st->done) {
        st->done = 1;
        if (st->errflag) {
            st->numerical = 1;
            st->final_it = num_iter - 1;
        } else {
            st->final_it = num_iter;
        }
    }
}

// Ybar[i, c] = sum_j P[i, j] Y[j, c] / (sum_j P[i, j] + 1e-32),  P[i, j] = u[i] K[i, j] v[j]     (:55-56)
__global__ void __launch_bounds__(256) ot_barycentric_kernel(const double* __restrict__ K, const double* __restrict__ ubuf,
                                                             const double* __restrict__ vbuf, const double* __restrict__ Y,
                                                             int ns, int nt, int C, const OtState* st,
                                                             double* __restrict__ ybar) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= ns) return;
    const int par = st->final_it & 1;
    const double ui = ubuf[(long long)par * ns + row];
    const double* v = vbuf + (long long)par * nt;
    const double* kr = K + (long long)row * nt;
    double sp = 0.0, sy[OT_MAXC];
    for (int c = 0; c < OT_MAXC; ++c) sy[c] = 0.0;
    for (int j = lane; j < nt; j += 32) {
        const double p = (ui * kr[j]) * v[j];
        sp += p;
        for (int c = 0; c < OT_MAXC; ++c)
            if (c < C) sy[c] = fma(p, Y[(long long)j * C + c], sy[c]);
    }
    sp = warp_sum(sp);
    for (int c = 0; c < OT_MAXC; ++c) sy[c] = warp_sum(sy[c]);
    if (lane == 0)
        for (int c = 0; c < C; ++c) ybar[(long long)row * C + c] = sy[c] / (sp + 1e-32);
}

// ---------------------------------------------------------------------------------- fp64 polyfit of the targets
// moments of S series of n fp64 samples (element (i, s) at x[i * S + s]: the [n, C] layout of X and Ybar);
// one block per series, fixed-order reduction.  Same sums as poly.cu's accumulate<DEG>, generic degree.
__global__ void __launch_bounds__(256) moments_f64_kernel(const double* __restrict__ x, const double* __restrict__ y,
                                                          long long n, int S, int deg, double* __restrict__ moments) {
    __shared__ double red[8][3 * HSR_MAX_POLY_DEG + 2];
    const int s = blockIdx.x, M = 3 * deg + 2;
    double acc[3 * HSR_MAX_POLY_DEG + 2];
    for (int j = 0; j < M; ++j) acc[j] = 0.0;
    for (long long i = threadIdx.x; i < n; i += 256) {
        const double xv = x[i * S + s], yv = y[i * S + s];
        if (isfinite(xv) && isfinite(yv)) {
            double pw[HSR_MAX_POLY_DEG + 1];
            pw[0] = 1.0;
            for (int j = 1; j <= deg; ++j) pw[j] = pw[j - 1] * xv;
            acc[0] += 1.0;
            acc[1] += xv;
            for (int j = 2; j <= 2 * deg; ++j) acc[j] = fma(pw[j / 2], pw[j - j / 2], acc[j]);
            acc[2 * deg + 1] += yv;
            for (int j = 1; j <= deg; ++j) acc[2 * deg + 1 + j] = fma(pw[j], yv, acc[2 * deg + 1 + j]);
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j = 0; j < M; ++j) {
        const double t = warp_sum(acc[j]);
        if (lane == 0) red[warp][j] = t;
    }
    __syncthreads();
    if (threadIdx.x < M) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
        moments[(long long)s * M + threadIdx.x] = t;
    }
}

__global__ void ot_info_kernel(const OtState* s, double* o) {
    o[0] = (double)s->final_it;
    o[1] = s->err;
    o[2] = (double)s->err_it;
    o[3] = (double)s->numerical;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int col_chunks(int ns) {
    int c = ns / 128;
    if (c < 1) c = 1;
    if (c > 32) c = 32;
    return c;
}

}  // namespace

constexpr int COMPACT_ROWS = 4096;

size_t compact_workspace(long long n) {
    if (n < 0) return 0;
    const long long nb = (n + COMPACT_ROWS - 1) / COMPACT_ROWS;
    return align_up((size_t)(nb + 1) * sizeof(unsigned int), 256) + align_up((size_t)(nb + 1) * sizeof(long long), 256);
}

int compact_finite_rows_impl(const float* img, const uint8_t* mask, long long n, int C, void* workspace, int* idx,
                             long long* count, cudaStream_t stream) {
    HSR_REQUIRE(img && workspace && idx && count, HSR_EINVAL, "null img / workspace / idx / count pointer");
    HSR_REQUIRE(n >= 0 && n < 2147483647LL && C >= 1 && C <= OT_MAXC, HSR_ERANGE, "bad n = %lld or C = %d (C <= %d)", n,
                C, OT_MAXC);
    const int nb = (int)((n + COMPACT_ROWS - 1) / COMPACT_ROWS);
    unsigned int* bc = reinterpret_cast<unsigned int*>(workspace);
    long long* bb = reinterpret_cast<long long*>(reinterpret_cast<unsigned char*>(workspace) +
                                                 align_up((size_t)(nb + 1) * sizeof(unsigned int), 256));
    if (nb > 0) compact_count_kernel<<<nb, 256, 0, stream>>>(img, mask, n, C, COMPACT_ROWS, bc);
    compact_scan_kernel<<<1, 32, 0, stream>>>(bc, nb, bb, count);
    if (nb > 0) compact_scatter_kernel<<<nb, 256, 0, stream>>>(img, mask, n, C, COMPACT_ROWS, bb, idx);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int gather_rows_impl(const float* img, const int* idx, const long long* sel, long long ns, int C, double* out,
                     cudaStream_t stream) {
    HSR_REQUIRE(img && idx && sel && out, HSR_EINVAL, "null img / idx / sel / out pointer");
    HSR_REQUIRE(ns >= 0 && C >= 1 && C <= OT_MAXC, HSR_ERANGE, "bad ns = %lld or C = %d", ns, C);
    if (ns == 0) return HSR_OK;
    gather_rows_kernel<<<(unsigned int)((ns * C + 255) / 256), 256, 0, stream>>>(img, idx, sel, ns, C, out);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

size_t sinkhorn_workspace(int ns, int nt) {
    if (ns < 1 || nt < 1) return 0;
    size_t b = align_up(sizeof(OtState), 256);
    b += align_up((size_t)ns * nt * 8, 256);                 // K
    b += align_up((size_t)2 * ns * 8, 256);                  // u (two iterations)
    b += align_up((size_t)2 * nt * 8, 256);                  // v
    b += align_up((size_t)nt * 8, 256);                      // v-update: per-block error terms and flags
    b += align_up((size_t)OT_PARTS_MAX * nt * 8, 256);       // column-pass partials (one row per chunk / per CTA)
    return b;
}

int sinkhorn_barycentric_impl(const double* X, const double* Y, int ns, int nt, int C, double reg, int num_iter_max,
                              double stop_thr, void* workspace, double* ybar, double* info, cudaStream_t stream) {
    HSR_REQUIRE(X && Y && workspace && ybar, HSR_EINVAL, "null X / Y / workspace / ybar pointer");
    HSR_REQUIRE(ns >= 1 && nt >= 1 && C >= 1 && C <= OT_MAXC, HSR_ERANGE, "bad ns = %d, nt = %d or C = %d", ns, nt, C);
    HSR_REQUIRE(reg > 0.0 && num_iter_max >= 0, HSR_EINVAL, "reg must be > 0 and numItermax >= 0");
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, HSR_EALIGN, "workspace not 256-byte aligned");
    unsigned char* w = reinterpret_cast<unsigned char*>(workspace);
    OtState* st = reinterpret_cast<OtState*>(w);
    w += align_up(sizeof(OtState), 256);
    double* K = reinterpret_cast<double*>(w);
    w += align_up((size_t)ns * nt * 8, 256);
    double* u = reinterpret_cast<double*>(w);
    w += align_up((size_t)2 * ns * 8, 256);
    double* v = reinterpret_cast<double*>(w);
    w += align_up((size_t)2 * nt * 8, 256);
    double* e2part = reinterpret_cast<double*>(w);
    int* badpart = reinterpret_cast<int*>(e2part + (nt + VUP_COLS - 1) / VUP_COLS + 8);
    w += align_up((size_t)nt * 8, 256);
    double* partial = reinterpret_cast<double*>(w);

    const int nmax = ns > nt ? ns : nt;
    ot_init_kernel<<<(nmax + 255) / 256, 256, 0, stream>>>(u, v, ns, nt, st);
    dim3 gk((nt + 255) / 256, (ns + 15) / 16);
    ot_kernel_matrix<<<gk, 256, 0, stream>>>(X, Y, ns, nt, C, reg, K);
    const int nchunks = col_chunks(ns);
    const int rpc = (ns + nchunks - 1) / nchunks;
    dim3 gc((nt + COL_THREADS - 1) / COL_THREADS, nchunks);
    const int vblocks = (nt + VUP_COLS - 1) / VUP_COLS;
    const double a = 1.0 / ns, b = 1.0 / nt;   // a = np.full(ns, 1.0 / ns), b = np.full(nt, 1.0 / nt)  (:49-50)
    const double inv_a = 1.0 / a;              // Kp = (1 / a).reshape(-1, 1) * K
    // fused path: whole rows fit the shared-memory ring (four rows) and rows are 16-byte multiples
    const size_t fuse_smem = 256 + (size_t)FUSE_NST * nt * 8;
    int fgrid = device_sm_count();
    if (fgrid > OT_PARTS_MAX) fgrid = OT_PARTS_MAX;
    if (fgrid > ns) fgrid = ns;
    const bool fused = (nt % 2 == 0) && nt <= FUSE_NCMAX * FUSE_THREADS && fuse_smem <= (size_t)device_max_smem_optin();
    if (fused)
    {
        static int set__[HSR_MAX_DEVICES];
        HSR_CUDA(ensure_dynamic_smem(ot_fused_kernel, (int)fuse_smem, set__));
    }
    int nparts = nchunks;
    bool looped = false;
    if (fused && num_iter_max > 0) {
        // Device-side loop: a CUDA-graph WHILE node whose body is {v-update, fused sweep, step}; the step kernel ends
        // the loop as soon as the marginal error is below stopThr (or after numItermax iterations), so nothing is
        // enqueued for iterations that never run.  The first column pass (u_0) fills nchunks partial rows; the rest
        // of the fgrid rows the body reads are zeroed once.
        HSR_CUDA(cudaMemsetAsync(partial + (size_t)nchunks * nt, 0, (size_t)(fgrid - nchunks) * nt * 8, stream));
        ot_colpass_kernel<<<gc, COL_THREADS, (size_t)rpc * 8, stream>>>(K, u, ns, nt, 0, rpc, partial, st);
        cudaGraph_t graph = nullptr, body = nullptr, captured = nullptr;
        cudaGraphExec_t exec = nullptr;
        cudaStream_t cap = nullptr;
        cudaGraphConditionalHandle handle;
        bool ok = cudaGraphCreate(&graph, 0) == cudaSuccess &&
                  cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault) == cudaSuccess;
        if (ok) {
            cudaGraphNodeParams np = {};
            np.type = cudaGraphNodeTypeConditional;
            np.conditional.handle = handle;
            np.conditional.type = cudaGraphCondTypeWhile;
            np.conditional.size = 1;
            cudaGraphNode_t node;
            ok = cudaGraphAddNode(&node, graph, nullptr, 0, &np) == cudaSuccess;
            if (ok) body = np.conditional.phGraph_out[0];
        }
        ok = ok && cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking) == cudaSuccess;
        if (ok && cudaStreamBeginCaptureToGraph(cap, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            ot_vupdate_kernel<<<vblocks, VUP_THREADS, 0, cap>>>(partial, fgrid, ns, nt, -1, b, stop_thr, v, e2part, badpart, st);
            ot_fused_kernel<<<fgrid, FUSE_THREADS, fuse_smem, cap>>>(K, v, u, ns, nt, -1, inv_a, partial, st);
            ot_step_kernel<<<1, 32, 0, cap>>>(st, handle, num_iter_max);
            ok = cudaStreamEndCapture(cap, &captured) == cudaSuccess;
        } else {
            ok = false;
        }
        ok = ok && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
        if (ok) {
            ok = cudaGraphLaunch(exec, stream) == cudaSuccess;
            looped = ok;
        }
        if (exec) cudaGraphExecDestroy(exec);   // in-flight launches complete; resources are released afterwards
        if (graph) cudaGraphDestroy(graph);
        if (cap) cudaStreamDestroy(cap);
        if (!looped) {
            (void)cudaGetLastError();           // fall back to the enqueue-everything loop below (it = 0 redone: idempotent)
        }
    }
    for (int it = 0; !looped && it < num_iter_max; ++it) {
        if (!fused || it == 0) {
            ot_colpass_kernel<<<gc, COL_THREADS, (size_t)rpc * 8, stream>>>(K, u, ns, nt, it, rpc, partial, st);
            nparts = nchunks;
        }
        ot_vupdate_kernel<<<vblocks, VUP_THREADS, 0, stream>>>(partial, nparts, ns, nt, it, b, stop_thr, v, e2part, badpart, st);
        if (fused) {
            // row pass of `it` + column pass of `it + 1` in one sweep of K (its partials feed the next v-update)
            ot_fused_kernel<<<fgrid, FUSE_THREADS, fuse_smem, stream>>>(K, v, u, ns, nt, it, inv_a, partial, st);
            nparts = fgrid;
        } else {
            ot_rowpass_kernel<<<(ns + 7) / 8, 256, 0, stream>>>(K, v, ns, nt, it, inv_a, u, st);
        }
    }
    ot_finish_kernel<<<1, 32, 0, stream>>>(num_iter_max, st);
    ot_barycentric_kernel<<<(ns + 7) / 8, 256, 0, stream>>>(K, u, v, Y, ns, nt, C, st, ybar);
    HSR_CUDA(cudaGetLastError());
    if (info) {  // {final iteration, last evaluated error, iteration it was evaluated at, numerical-error flag}
        ot_info_kernel<<<1, 1, 0, stream>>>(st, info);
        HSR_CUDA(cudaGetLastError());
    }
    return HSR_OK;
}

int polyfit_f64_moments_impl(const double* x, const double* y, long long n, int S, int deg, double* moments,
                             cudaStream_t stream) {
    HSR_REQUIRE(x && y && moments, HSR_EINVAL, "null x / y / moments pointer");
    HSR_REQUIRE(n >= 0 && S >= 1 && S <= 65535, HSR_ERANGE, "bad n = %lld or S = %d", n, S);
    HSR_REQUIRE(deg >= 1 && deg <= HSR_MAX_POLY_DEG, HSR_ERANGE, "deg = %d outside [1, %d]", deg, HSR_MAX_POLY_DEG);
    moments_f64_kernel<<<S, 256, 0, stream>>>(x, y, n, S, deg, moments);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

// ---------------------------------------------------------------------------- affine colour transfer
// s2_emit/color.py:103-115 — W = lstsq([X 1], Ybar) (A = W[:C], t = W[C]) and out[mask] = clip(X @ A + t, 0, 1).
namespace {

constexpr int AFF_THREADS = 256;
constexpr int AFF_MAXD = OT_MAXC + 1;

// One CTA: normal equations G = [X 1]^T [X 1] ((C+1)^2) and R = [X 1]^T Ybar ((C+1) x C) in fp64, reduced in a fixed
// order (per-thread strided sums -> warp shuffles -> 8 warp partials added in order), then Gauss-Jordan with partial
// pivoting by thread 0.  W is [(C+1), C] row-major.  A singular system (degenerate samples) yields NaN, like a
// failed fit; numpy's lstsq would return the minimum-norm solution there.
__global__ void __launch_bounds__(AFF_THREADS) affine_fit_kernel(const double* __restrict__ X, const double* __restrict__ Yb,
                                                                 long long ns, int C, double* __restrict__ W) {
    const int D = C + 1;
    const int nG = D * D, nR = D * C, nT = nG + nR;
    __shared__ double part[AFF_THREADS / 32][AFF_MAXD * AFF_MAXD + AFF_MAXD * OT_MAXC];
    __shared__ double M[AFF_MAXD][AFF_MAXD + OT_MAXC];
    double acc[AFF_MAXD * AFF_MAXD + AFF_MAXD * OT_MAXC];
#pragma unroll
    for (int i = 0; i < AFF_MAXD * AFF_MAXD + AFF_MAXD * OT_MAXC; ++i) acc[i] = 0.0;
    for (long long r = threadIdx.x; r < ns; r += AFF_THREADS) {
        double xa[AFF_MAXD], yb[OT_MAXC];
#pragma unroll
        for (int c = 0; c < OT_MAXC; ++c) {
            xa[c] = c < C ? X[r * C + c] : 0.0;
            yb[c] = c < C ? Yb[r * C + c] : 0.0;
        }
        xa[C] = 1.0;
#pragma unroll
        for (int i = 0; i < AFF_MAXD; ++i) {
            if (i >= D) break;
#pragma unroll
            for (int j = 0; j < AFF_MAXD; ++j)
                if (j < D) acc[i * AFF_MAXD + j] += xa[i] * xa[j];
#pragma unroll
            for (int j = 0; j < OT_MAXC; ++j)
                if (j < C) acc[AFF_MAXD * AFF_MAXD + i * OT_MAXC + j] += xa[i] * yb[j];
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < AFF_MAXD * AFF_MAXD + AFF_MAXD * OT_MAXC; ++i) {
        const double v = warp_sum(acc[i]);
        if (lane == 0) part[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        (void)nT;
        (void)nG;
        (void)nR;
        for (int i = 0; i < D; ++i) {
            for (int j = 0; j < D; ++j) {
                double v = 0.0;
                for (int w = 0; w < AFF_THREADS / 32; ++w) v += part[w][i * AFF_MAXD + j];
                M[i][j] = v;
            }
            for (int j = 0; j < C; ++j) {
                double v = 0.0;
                for (int w = 0; w < AFF_THREADS / 32; ++w) v += part[w][AFF_MAXD * AFF_MAXD + i * OT_MAXC + j];
                M[i][D + j] = v;
            }
        }
        for (int col = 0; col < D; ++col) {
            int piv = col;
            for (int r = col + 1; r < D; ++r)
                if (fabs(M[r][col]) > fabs(M[piv][col])) piv = r;
            if (piv != col)
                for (int j = 0; j < D + C; ++j) {
                    const double t = M[col][j];
                    M[col][j] = M[piv][j];
                    M[piv][j] = t;
                }
            const double inv = 1.0 / M[col][col];
            for (int j = 0; j < D + C; ++j) M[col][j] *= inv;
            for (int r = 0; r < D; ++r) {
                if (r == col) continue;
                const double f = M[r][col];
                for (int j = 0; j < D + C; ++j) M[r][j] -= f * M[col][j];
            }
        }
        for (int i = 0; i < D; ++i)
            for (int j = 0; j < C; ++j) W[i * C + j] = M[i][D + j];
    }
}

// out = float32 copy of rgb; where mask: float32(clip(float64(x) @ A + t, lo, hi)) (NaN stays NaN, as np.clip).
__global__ void __launch_bounds__(256) affine_apply_kernel(const float* __restrict__ rgb, const double* __restrict__ W,
                                                           const uint8_t* __restrict__ mask, long long n, int C,
                                                           double lo, double hi, float* __restrict__ out) {
    __shared__ double sW[AFF_MAXD * OT_MAXC];
    if (threadIdx.x < (C + 1) * C) sW[threadIdx.x] = W[threadIdx.x];
    __syncthreads();
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        float x[OT_MAXC];
#pragma unroll
        for (int c = 0; c < OT_MAXC; ++c)
            if (c < C) x[c] = rgb[p * C + c];
        if (mask == nullptr || mask[p]) {
#pragma unroll
            for (int j = 0; j < OT_MAXC; ++j) {
                if (j >= C) break;
                double v = 0.0;
#pragma unroll
                for (int c = 0; c < OT_MAXC; ++c)
                    if (c < C) v = fma((double)x[c], sW[c * C + j], v);      // row of x times column j of A
                v += sW[C * C + j];
                v = v < lo ? lo : (v > hi ? hi : v);
                out[p * C + j] = (float)v;
            }
        } else {
#pragma unroll
            for (int c = 0; c < OT_MAXC; ++c)
                if (c < C) out[p * C + c] = x[c];
        }
    }
}

}  // namespace

int affine_fit_impl(const double* X, const double* Ybar, long long ns, int C, double* W, cudaStream_t stream) {
    HSR_REQUIRE(X && Ybar && W, HSR_EINVAL, "null X / Ybar / W pointer");
    HSR_REQUIRE(ns >= 1 && C >= 1 && C <= OT_MAXC, HSR_ERANGE, "ns = %lld, C = %d outside [1, inf) x [1, %d]", ns, C, OT_MAXC);
    affine_fit_kernel<<<1, AFF_THREADS, 0, stream>>>(X, Ybar, ns, C, W);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int affine_apply_impl(const float* rgb, const double* W, const uint8_t* mask, long long n, int C, float lo, float hi,
                      float* out, cudaStream_t stream) {
    HSR_REQUIRE(rgb && W && out, HSR_EINVAL, "null rgb / W / out pointer");
    HSR_REQUIRE(n >= 0 && C >= 1 && C <= OT_MAXC, HSR_ERANGE, "n = %lld, C = %d outside the supported range", n, C);
    if (n == 0) return HSR_OK;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)device_sm_count() * 8;
    affine_apply_kernel<<<(unsigned int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(rgb, W, mask, n, C, (double)lo,
                                                                                       (double)hi, out);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

}  // namespace hsr
