// glt_stream.cu — kernels 1 and 2 of the hot path: GLT-indexed ortho gather of the
// band-interleaved cube (bit-exact copy/fill) and the fused gather + SRF contraction.
//
// One persistent CTA per SM, warp-specialised around a ring of shared-memory stages, one
// 32-pixel ortho tile per stage:
//   PRODUCER warps (nprod; producer w owns stages w, w + nprod, ...): lane i owns pixel i of the
//   tile.  The GLT entries come from a per-producer shared-memory ring filled by 16-byte cp.async
//   copies GLT_DEPTH tiles ahead (when the GLT planes are contiguous and 16-byte aligned; otherwise
//   each lane loads its own entries).  The lanes evaluate the validity rule of
//   EMIT_data/emit_proj.py:691-703, then MERGE lanes whose source pixels are the same or adjacent
//   in memory (q[l] - q[l-1] in {0, 1}) into runs: one bulk copy per run brings the 16-byte
//   aligned window covering the run's spectra (n * 1140 B for 285 bands) into the stage, runs
//   packed back to back.  A 25-degree GLT needs ~13 copies per tile instead of 32, an identity
//   GLT one.
//   CONSUMER warps (CPS per stage): wait on the stage's mbarrier and either re-align the spectra
//   into 16-byte vector stores of the ortho cube (emit_proj.py:981-982; each warp half of the
//   pixels), or run the SRF contraction of s2_emit/synth.py:41-43 with one lane per pixel (each
//   warp half of the non-finite scan and a load-balanced half of the S2 bands), or both.
// No data-path instruction touches the raw cube outside the TMA unit.
#include "hsr_common.cuh"

namespace hsr {

namespace {

constexpr int TILE = HSR_TILE_PX;  // ortho pixels per tile == lanes of a warp
constexpr int MAX_STAGES = 5;
constexpr int MAX_PRODUCERS = 5;
constexpr int MAX_CPS = 4;  // consumer warps per stage: 4 for the SRF contraction, 2 when the cube is materialised
__host__ __device__ constexpr int cps_of(int mode) { return (mode & 1) ? 2 : 4; }
__host__ __device__ constexpr int nthreads_of(int mode) { return 32 * (MAX_PRODUCERS + cps_of(mode) * MAX_STAGES); }
constexpr int GLT_DEPTH = 4;  // GLT tiles staged ahead of the gather, per producer warp
constexpr int MAXK = HSR_MAX_SRF_BANDS;

constexpr int MODE_COPY = 1;
constexpr int MODE_SRF = 2;
constexpr int MODE_Q16 = 4;  // quantised band-sequential uint16 cube + black mask (tile export), no fp32 cube

constexpr long long MAX_PIXELS = 2147483584LL;  // 2^31 - 64: pixel indices are 32-bit in the kernels

constexpr int META_FILL = -1;  // pixel inside the grid, GLT invalid -> fill value
constexpr int META_OOB = -2;   // lane beyond the end of the grid (last tile only)

struct StreamParams {
    const float* raw;
    long long raw_h, raw_w, raw_pix_stride;
    int bands;
    int transpose;
    int identity;  // 1: no GLT, source pixel == output pixel (un-fused SRF)
    // hsr_raw_view_t: `raw` holds only slow-axis indices [win_lo, win_lo + win_n) of the cube (rows; columns when
    // transposed) — per-slab staging of a mosaic, row-range uploads; and / or the ortho grid is a stack of
    // independent tiles of batch_out_rows rows whose GLT entries index their own raw tile of batch_raw_rows rows
    unsigned int win_lo, win_n;
    int batch_out_rows, batch_raw_rows;
    int has_view;  // diag has a fourth word (valid entries whose source lies outside the window)
    int merge;     // 1: raw_pix_stride == bands, adjacent source pixels are contiguous -> run merging
    const int32_t* glt_x;
    const int32_t* glt_y;
    long long out_w, glt_row_stride, npix, ntiles;
    int glt_ring;  // GLT planes contiguous and 16-byte aligned -> staged ahead in shared memory by cp.async
    float fill;
    float* ortho;
    long long out_pix_stride;
    uint8_t* valid;
    unsigned long long* diag;
    const float* W;
    const float* fill_out;
    int K;
    float* bands_out;
    long long plane_stride;
    // MODE_Q16: tiles_helpers/utils.py:357-371 (uint16 quantisation) and :201-220 (is_black_mask) of the ortho pixel
    unsigned short* q16;  // [bands][q16_plane_stride] band-sequential
    long long q16_plane_stride;
    float q_scale, q_nodata, q_hi;
    int q_has_nodata;
    unsigned short q_nd, q_fill;  // nodata code; quantised fill value (what an invalid GLT pixel gets)
    int q16_pair;                 // planes 4-byte aligned with an even stride: two pixels per lane, 4-byte stores
    uint8_t* black;               // nullable [npix]
    float b_nodata_tol, b_masked, b_masked_tol, b_zero_tol;
    int black_fill;               // bit 0 / 1 / 2: a fill pixel satisfies the nodata / masked / zero rule
    uint8_t* fit_mask;  // nullable: valid & all_k isfinite(bands_out[k]) & (bands_out[gate_k] > gate_gt)
    int gate_k;
    float gate_gt;
    int stage_f4;   // float4 per stage
    int nstage;
    int nprod;
    int wt_pitch;   // floats per row of the transposed weight table in smem
    int bank_step;  // odd: bank distance (in words, mod 32) the producers put between consecutive lanes
    unsigned long long raw_lo, raw_hi;  // byte range of the raw cube that may be read
};

struct SmemHeader {
    uint64_t full[MAX_STAGES];
    uint64_t empty[MAX_STAGES];
    int meta[MAX_STAGES][TILE];  // >= 0: word offset of the pixel's spectrum inside its stage
    int glt[MAX_PRODUCERS][GLT_DEPTH][2][TILE];
    int fill_f4[MAX_STAGES];                // float4 of the stage the tile's runs occupy (gaps included)
    int tile_id[MAX_STAGES];                // tile the stage holds (-1: no more tiles) — see producer_fills()
    int krun[2][MAXK];                      // first band (multiple of 4) / end of the non-zero run of each folded response
    unsigned int badbits[MAX_STAGES][MAX_CPS];  // per consumer warp: its half of the stage holds a non-finite word
    unsigned int fm_word[MAX_STAGES][MAX_CPS];  // per consumer warp: fit-mask bits of its share of the S2 bands
    unsigned int bk_word[MAX_STAGES][MAX_CPS][3];  // per consumer warp: black-mask rule bits over its share of the bands
    int4 kparam[MAX_CPS][MAXK];  // per consumer warp of a stage, its S2 bands (balanced by run length):
                             // {k, b0 (first band, multiple of 4), b1v (end of the float4 part), b1 (end)}
    int kcount[MAX_CPS];
    float fill_out[MAXK];
};
static_assert(offsetof(SmemHeader, glt) % 16 == 0, "GLT ring must be 16-byte aligned for 16-byte cp.async");
static_assert(offsetof(SmemHeader, kparam) % 16 == 0, "kparam is read with 16-byte loads");

__host__ __device__ inline int header_bytes() { return (int)((sizeof(SmemHeader) + 127) / 128 * 128); }

// Fused SRF without a materialised cube: a tile that holds no valid pixel is finished BY ITS PRODUCER (K fill stores, a
// zero fit-mask word) and never enters the ring — a nodata tile through the ring costs a whole stage round trip
// (~1 us of a stage's time while moving no bytes; 43 % of a rotated granule's tiles).  The stage then no longer holds
// "tile number `use`" of a fixed sequence, so the producer passes the tile id through shared memory and ends the
// sequence with -1.  Needs one producer per stage (a single fill counter gives the barrier parity).
template <int MODE>
__device__ __forceinline__ bool producer_fills(const StreamParams& P) {
    return MODE == MODE_SRF && P.nprod == P.nstage && !P.identity;
}

__device__ __forceinline__ void glt_cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void glt_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void glt_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int D>
__device__ __forceinline__ float4 realign(const float4 a, const float4 b) {
    if (D == 0) return a;
    if (D == 1) return make_float4(a.y, a.z, a.w, b.x);
    if (D == 2) return make_float4(a.z, a.w, b.x, b.y);
    return make_float4(a.w, b.x, b.y, b.z);
}

// Copy nfull aligned float4 of one pixel: source window words start D words into w4[0].
template <int D>
__device__ __forceinline__ void copy_pixel_f4(const float4* __restrict__ w4, float4* __restrict__ dst4, int nfull,
                                               int lane) {
    for (int base = 0; base < nfull; base += 96) {
        const int j0 = base + lane, j1 = j0 + 32, j2 = j0 + 64;
        const bool p0 = j0 < nfull, p1 = j1 < nfull, p2 = j2 < nfull;
        float4 a0, b0, a1, b1, a2, b2;
        a0 = b0 = a1 = b1 = a2 = b2 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p0) { a0 = w4[j0]; if (D) b0 = w4[j0 + 1]; }
        if (p1) { a1 = w4[j1]; if (D) b1 = w4[j1 + 1]; }
        if (p2) { a2 = w4[j2]; if (D) b2 = w4[j2 + 1]; }
        if (p0) __stcs(dst4 + j0, realign<D>(a0, b0));
        if (p1) __stcs(dst4 + j1, realign<D>(a1, b1));
        if (p2) __stcs(dst4 + j2, realign<D>(a2, b2));
    }
}

// Consumer, ortho materialisation: warp `half` walks pixels [16*half, 16*half + 16) of the tile; per
// pixel the lanes stream 16-byte stores (head/tail words of the unaligned 1140-byte record are scalar).
template <int CPS>
__device__ __forceinline__ void copy_tile(const StreamParams& P, const float4* __restrict__ st4, int m, long long tile,
                                          int lane, int half) {
    const int B = P.bands;
    const float fillv = P.fill;
    const float4 fill4 = make_float4(fillv, fillv, fillv, fillv);
    const int k0 = half * (TILE / CPS);
    for (int k = k0; k < k0 + TILE / CPS; ++k) {
        const int mk = __shfl_sync(0xffffffffu, m, k);
        if (mk == META_OOB) break;
        const long long p = tile * TILE + k;
        float* dst = P.ortho + p * P.out_pix_stride;
        const int dp = (int)((reinterpret_cast<uintptr_t>(dst) >> 2) & 3);
        int h = (4 - dp) & 3;
        if (h > B) h = B;
        const int nfull = (B - h) >> 2;
        const int t = (B - h) & 3;
        float4* dst4 = reinterpret_cast<float4*>(dst + h);
        if (mk >= 0) {
            const float* wf = reinterpret_cast<const float*>(st4);  // spectrum = wf[mk .. mk + B)
            const int s = mk + h;
            const float4* w4 = st4 + (s >> 2);
            switch (s & 3) {
                case 0: copy_pixel_f4<0>(w4, dst4, nfull, lane); break;
                case 1: copy_pixel_f4<1>(w4, dst4, nfull, lane); break;
                case 2: copy_pixel_f4<2>(w4, dst4, nfull, lane); break;
                default: copy_pixel_f4<3>(w4, dst4, nfull, lane); break;
            }
            if (lane < h) __stcs(dst + lane, wf[mk + lane]);
            const int tl = lane - 8;
            if (tl >= 0 && tl < t) __stcs(dst + h + 4 * nfull + tl, wf[s + 4 * nfull + tl]);
        } else {
            for (int j = lane; j < nfull; j += 32) __stcs(dst4 + j, fill4);
            if (lane < h) __stcs(dst + lane, fillv);
            const int tl = lane - 8;
            if (tl >= 0 && tl < t) __stcs(dst + h + 4 * nfull + tl, fillv);
        }
    }
}

// acc += {a, b} * {0, 0} as one packed FFMA2: stays 0 unless a or b is NaN / Inf
__device__ __forceinline__ void scan2(unsigned long long& acc, float a, float b) {
    unsigned long long ab;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ab) : "f"(a), "f"(b));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(ab), "l"(0ull));
}

// Precise per-lane non-finite test of one spectrum (slow path of the scan): aligned window w4,
// spectrum = words [sp, sp + B).
__device__ __noinline__ bool spectrum_nonfinite(const float4* __restrict__ w4, int sp, int B) {
    const int end = sp + B;
    const int n4 = (end + 3) >> 2;
    float z = 0.f;
    for (int i = 0; i < n4; ++i) {
        const float4 v = w4[i];
        const int w = 4 * i;
        if (w + 0 >= sp && w + 0 < end) z = fmaf(v.x, 0.f, z);
        if (w + 1 >= sp && w + 1 < end) z = fmaf(v.y, 0.f, z);
        if (w + 2 >= sp && w + 2 < end) z = fmaf(v.z, 0.f, z);
        if (w + 3 >= sp && w + 3 < end) z = fmaf(v.w, 0.f, z);
    }
    return !(z == 0.f);
}

// Consumer, SRF contraction: lane l owns pixel l of the tile; the two warps of a stage split the work.
//   1. non-finite scan (0*x accumulates NaN iff any sample is NaN/Inf): in synth.py:41 a non-finite
//      sample under a ZERO weight still poisons the integral, so every one of the `bands` samples
//      counts.  Fast path: the pair sweeps the occupied part of the stage linearly (conflict-free
//      16-byte loads, packed FFMA2), half each, and exchanges one flag through shared memory and a
//      named barrier; only when some word is non-finite (possibly a neighbour's sample in a window
//      overhang, or stale data in a gap: false positives are harmless) do the lanes test their own
//      spectrum word by word;
//   2. per S2 band k of this warp's list, fp32 FMA chains over the contiguous non-zero run of
//      W[:,k]; pixels flagged by the scan take a dense chain over all bands instead (exact IEEE
//      propagation).
template <int CPS>
__device__ __forceinline__ void srf_tile(const StreamParams& P, SmemHeader* hd, const float* __restrict__ wt,
                                         const float4* __restrict__ st4, int m, long long tile, int lane, int stage,
                                         int half) {
    const bool ok = m >= 0;
    const int nk = hd->kcount[half];
    const int4* kp = hd->kparam[half];
    const long long p = tile * TILE + lane;
    if (__ballot_sync(0xffffffffu, ok) == 0u) {  // whole tile is fill (both warps of the pair agree)
        if (m != META_OOB) {
            for (int j = 0; j < nk; ++j) {
                const int k = kp[j].x;
                P.bands_out[(long long)k * P.plane_stride + p] = hd->fill_out[k];
            }
            if (P.fit_mask && half == 0) P.fit_mask[p] = 0;
        }
        return;
    }
    const int B = P.bands;
    const int sp = ok ? (m & 3) : 0;
    const float4* w4 = st4 + (ok ? (m >> 2) : 0);  // aligned window: spectrum = words [sp, sp + B)
    const float* xs = reinterpret_cast<const float*>(w4) + sp;

    // ---- 1. non-finite scan of this warp's part of the occupied stage (result needed only after step 2)
    const int n4 = hd->fill_f4[stage];
    const int per = (n4 + CPS - 1) / CPS;
    const int lo = half * per, hi = (lo + per < n4) ? lo + per : n4;
    unsigned long long zz0 = 0ull, zz1 = 0ull, zz2 = 0ull, zz3 = 0ull;
    int i = lo + lane;
    for (; i + 96 < hi; i += 128) {
        const float4 a = st4[i], b = st4[i + 32], c = st4[i + 64], d = st4[i + 96];
        scan2(zz0, a.x, a.y);
        scan2(zz1, a.z, a.w);
        scan2(zz2, b.x, b.y);
        scan2(zz3, b.z, b.w);
        scan2(zz0, c.x, c.y);
        scan2(zz1, c.z, c.w);
        scan2(zz2, d.x, d.y);
        scan2(zz3, d.z, d.w);
    }
    for (; i < hi; i += 32) {
        const float4 a = st4[i];
        scan2(zz0, a.x, a.y);
        scan2(zz1, a.z, a.w);
    }
    float y0, y1, y2, y3, y4, y5, y6, y7;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(y0), "=f"(y1) : "l"(zz0));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(y2), "=f"(y3) : "l"(zz1));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(y4), "=f"(y5) : "l"(zz2));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(y6), "=f"(y7) : "l"(zz3));
    const float z = ((y0 + y1) + (y2 + y3)) + ((y4 + y5) + (y6 + y7));

    // ---- 2. per-band FMA over the non-zero run of the folded weights: 16-byte broadcast loads of four
    //         weights, four independent accumulators.  The run bounds are multiples of 4 inside the
    //         spectrum (zero weights pad them); the rare tail past bands & ~3 is scalar.  Independent of the
    //         scan, so the two interleave; pixels the scan flags are redone below.
    bool fit = ok;  // this warp's share of the fit mask: my bands are finite (and the gate band > gate_gt)
    for (int j = 0; j < nk; ++j) {
        const int4 kq = kp[j];
        const int k = kq.x, b0 = kq.y, b1v = kq.z, b1 = kq.w;
        const float* wk = wt + k * P.wt_pitch;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 2
        for (int b = b0; b < b1v; b += 4) {
            const float4 w = *reinterpret_cast<const float4*>(wk + b);
            a0 = fmaf(xs[b], w.x, a0);
            a1 = fmaf(xs[b + 1], w.y, a1);
            a2 = fmaf(xs[b + 2], w.z, a2);
            a3 = fmaf(xs[b + 3], w.w, a3);
        }
        for (int b = b1v; b < b1; ++b) a0 = fmaf(xs[b], wk[b], a0);
        float r = (a0 + a1) + (a2 + a3);
        if (!ok) r = hd->fill_out[k];
        if (m != META_OOB) P.bands_out[(long long)k * P.plane_stride + p] = r;
        fit = fit && finite_f32(r) && (k != P.gate_k || r > P.gate_gt);
    }

    // ---- 3. ONE exchange per tile: "my part of the stage holds a non-finite word" and my fit-mask bits.  The
    //         barrier is free: a consumer warp is bound to its stage, and the stage is only refilled once all CPS
    //         warps have released it anyway.
    {
        const unsigned int mine_bad = __ballot_sync(0xffffffffu, !(z == 0.f));
        const unsigned int mine_fit = __ballot_sync(0xffffffffu, fit);
        if (lane == 0) {
            hd->badbits[stage][half] = mine_bad;
            hd->fm_word[stage][half] = mine_fit;
        }
    }
    named_bar_sync(1 + stage, 32 * CPS);
    unsigned int any = 0u;
#pragma unroll
    for (int c = 0; c < CPS; ++c) any |= hd->badbits[stage][c];
    if (any != 0u) {
        // rare (uniform across the stage's warps): some word of the stage is non-finite, possibly a neighbour's
        // sample in a window overhang or stale data in a gap.  Test my own spectrum word by word and redo flagged
        // pixels densely over ALL samples so that IEEE propagation matches synth.py:41 exactly (NaN anywhere or
        // Inf under a zero weight -> NaN; Inf under a non-zero weight -> +-Inf).
        const bool bad = ok && spectrum_nonfinite(w4, sp, B);
        if (bad) {
            fit = true;
            for (int j = 0; j < nk; ++j) {
                const int k = kp[j].x;
                const float* wk = wt + k * P.wt_pitch;
                float r = 0.f;
                for (int b = 0; b < B; ++b) r = fmaf(xs[b], wk[b], r);
                P.bands_out[(long long)k * P.plane_stride + p] = r;
                fit = fit && finite_f32(r) && (k != P.gate_k || r > P.gate_gt);
            }
        }
        if (P.fit_mask) {  // nobody reads fm_word before the next barrier: rewrite it and exchange again
            const unsigned int mine_fit = __ballot_sync(0xffffffffu, fit);
            if (lane == 0) hd->fm_word[stage][half] = mine_fit;
            named_bar_sync(1 + stage, 32 * CPS);
        }
    }
    if (P.fit_mask && half == 0) {
        unsigned int word = 0xffffffffu;
#pragma unroll
        for (int c = 0; c < CPS; ++c) word &= hd->fm_word[stage][c];
        if (m != META_OOB) P.fit_mask[p] = (uint8_t)((word >> lane) & 1u);
    }
}

// Consumer, tile export: lane l owns pixel l of the tile, the CPS warps of a stage split the bands.  Every sample is
// quantised to uint16 (tiles_helpers/utils.py:357-371) and stored band-sequentially — 32 lanes x 2 bytes = one full
// 64-byte segment per band and tile — and the three is_black_mask rules (:201-220: all bands ~ nodata, all ~ masked
// value, all ~ 0) are tracked per lane while they can still hold, then ANDed across the warps through shared
// memory (same free barrier as the fit mask).  The fp32 ortho cube is never written.
template <int CPS>
__device__ __forceinline__ void q16_tile(const StreamParams& P, SmemHeader* hd, const float4* __restrict__ st4, int m,
                                         long long tile, int lane, int stage, int half) {
    const int B = P.bands;
    const long long p = tile * TILE + lane;
    const bool ok = m >= 0, inb = m != META_OOB;
    const int b0 = (int)((long long)B * half / CPS), b1 = (int)((long long)B * (half + 1) / CPS);
    unsigned short* out = P.q16 + p;
    const long long ps = P.q16_plane_stride;
    if (__ballot_sync(0xffffffffu, ok) == 0u) {  // whole tile is fill (all warps of the stage agree)
        if (inb) {
            for (int b = b0; b < b1; ++b) out[(long long)b * ps] = P.q_fill;
            if (P.black && half == 0) P.black[p] = P.black_fill ? 1 : 0;
        }
        return;
    }
    const float* xs = reinterpret_cast<const float*>(st4) + (ok ? m : 0);
    // rule bits still alive for my pixel: 1 nodata, 2 masked, 4 zero; fill pixels are constant across the bands
    unsigned int live = ok ? ((P.q_has_nodata ? 1u : 0u) | 6u) : (unsigned int)P.black_fill;
    const bool track = P.black != nullptr;
    // Branch-free inner loop: lanes without a source pixel read (valid) shared memory too and select the quantised
    // fill afterwards; lanes beyond the grid (last tile only) have their stores predicated off.  The rule bits are
    // evaluated per chunk of 8 bands, and only while some lane of the warp still has one alive (real spectra lose
    // all three within the first band or two).
    const int has_nd = P.q_has_nodata;
    const float nodata = P.q_nodata, scale = P.q_scale, hi = P.q_hi;
    const unsigned short nd = P.q_nd, qfill = P.q_fill;
    unsigned short* o = out + (long long)b0 * ps;
    for (int c0 = b0; c0 < b1; c0 += 8) {
        const int nb = b1 - c0 < 8 ? b1 - c0 : 8;
        if (track && __any_sync(0xffffffffu, ok && live != 0u)) {
            for (int j = 0; j < nb; ++j) {
                const float v = xs[c0 + j];
                if (ok && live) {
                    if (!close32(v, nodata, P.b_nodata_tol)) live &= ~1u;
                    if (!close32(v, P.b_masked, P.b_masked_tol)) live &= ~2u;
                    if (!(fabsf(v) < P.b_zero_tol)) live &= ~4u;
                }
            }
        }
        if (nb == 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const unsigned short q = quant_u16(xs[c0 + j], has_nd, nodata, scale, hi, nd);
                if (inb) *o = ok ? q : qfill;
                o += ps;
            }
        } else {
            for (int j = 0; j < nb; ++j) {
                const unsigned short q = quant_u16(xs[c0 + j], has_nd, nodata, scale, hi, nd);
                if (inb) *o = ok ? q : qfill;
                o += ps;
            }
        }
    }
    if (track) {
        const unsigned int w0 = __ballot_sync(0xffffffffu, live & 1u), w1 = __ballot_sync(0xffffffffu, live & 2u),
                           w2 = __ballot_sync(0xffffffffu, live & 4u);
        if (lane == 0) {
            hd->bk_word[stage][half][0] = w0;
            hd->bk_word[stage][half][1] = w1;
            hd->bk_word[stage][half][2] = w2;
        }
        named_bar_sync(1 + stage, 32 * CPS);
        if (half == 0) {
            unsigned int a0 = 0xffffffffu, a1 = 0xffffffffu, a2 = 0xffffffffu;
#pragma unroll
            for (int c = 0; c < CPS; ++c) {
                a0 &= hd->bk_word[stage][c][0];
                a1 &= hd->bk_word[stage][c][1];
                a2 &= hd->bk_word[stage][c][2];
            }
            if (inb) P.black[p] = (uint8_t)(((a0 | a1 | a2) >> lane) & 1u);
        }
    }
}

// Tile export, TWO pixels per lane (used when the planes allow 4-byte stores): lane l handles pixels 2 (l & 15) and
// 2 (l & 15) + 1 of the tile and every second band of the warp's share (band parity l >> 4), so one store instruction
// writes 2 bands x 64 bytes and the per-band loop overhead is shared by two samples (the one-pixel form was
// issue-bound at ~15 instructions per sample).  Bank check: spectrum p starts at bank 29 p (mod 32, bank-aware
// placement), so lanes read banks 26 (l & 15) + (l >> 4) + c — 32 distinct ones — and the same + 29 for the odd pixel.
template <int CPS>
__device__ __forceinline__ void q16_tile2(const StreamParams& P, SmemHeader* hd, const float4* __restrict__ st4, int m,
                                          long long tile, int lane, int stage, int half) {
    constexpr unsigned int FULL = 0xffffffffu;
    const int B = P.bands;
    const int b0 = (int)((long long)B * half / CPS), b1 = (int)((long long)B * (half + 1) / CPS);
    const int pp = lane & 15, hb = lane >> 4;
    const int m0 = __shfl_sync(FULL, m, 2 * pp), m1 = __shfl_sync(FULL, m, 2 * pp + 1);
    const bool ok0 = m0 >= 0, ok1 = m1 >= 0, in0 = m0 != META_OOB, in1 = m1 != META_OOB;
    const long long p = tile * TILE + 2 * pp;
    const long long ps = P.q16_plane_stride;
    if (__ballot_sync(FULL, m >= 0) == 0u) {  // whole tile is fill (all warps of the stage agree)
        const unsigned int f2 = (unsigned int)P.q_fill * 0x10001u;
        // (16-byte stores, four lanes per band and eight bands per instruction, cut the fill tiles' instructions by 8 x and
        // made the kernel SLOWER, 0.748 -> 0.774 ms: it is not issue-bound — see DESIGN.md 4.6)
        for (int c = b0 + hb; c < b1; c += 2) {
            unsigned short* o = P.q16 + (long long)c * ps + p;
            if (in0 && in1) *reinterpret_cast<unsigned int*>(o) = f2;
            else if (in0) *o = P.q_fill;
        }
        if (P.black && half == 0 && m != META_OOB) P.black[tile * TILE + lane] = P.black_fill ? 1 : 0;
        return;
    }
    const float* xs0 = reinterpret_cast<const float*>(st4) + (ok0 ? m0 : 0);
    const float* xs1 = reinterpret_cast<const float*>(st4) + (ok1 ? m1 : 0);
    // rule bits still alive (1 nodata, 2 masked, 4 zero) for my two pixels over MY bands; fill pixels are constant
    unsigned int live0 = ok0 ? ((P.q_has_nodata ? 1u : 0u) | 6u) : (unsigned int)P.black_fill;
    unsigned int live1 = ok1 ? ((P.q_has_nodata ? 1u : 0u) | 6u) : (unsigned int)P.black_fill;
    const bool track = P.black != nullptr;
    const int has_nd = P.q_has_nodata;
    const float nodata = P.q_nodata, scale = P.q_scale, hi = P.q_hi;
    const unsigned short nd = P.q_nd, qfill = P.q_fill;
    unsigned short* o = P.q16 + (long long)(b0 + hb) * ps + p;
    const long long ostep = 2 * ps;
    for (int c0 = b0 + hb; c0 < b1; c0 += 16) {               // chunks of 8 of my bands
        const int nb = (b1 - c0 + 1) / 2 < 8 ? (b1 - c0 + 1) / 2 : 8;
        if (track && __any_sync(FULL, (ok0 && live0 != 0u) || (ok1 && live1 != 0u))) {
            for (int j = 0; j < nb; ++j) {
                const float v0 = xs0[c0 + 2 * j], v1 = xs1[c0 + 2 * j];
                if (ok0 && live0) {
                    if (!close32(v0, nodata, P.b_nodata_tol)) live0 &= ~1u;
                    if (!close32(v0, P.b_masked, P.b_masked_tol)) live0 &= ~2u;
                    if (!(fabsf(v0) < P.b_zero_tol)) live0 &= ~4u;
                }
                if (ok1 && live1) {
                    if (!close32(v1, nodata, P.b_nodata_tol)) live1 &= ~1u;
                    if (!close32(v1, P.b_masked, P.b_masked_tol)) live1 &= ~2u;
                    if (!(fabsf(v1) < P.b_zero_tol)) live1 &= ~4u;
                }
            }
        }
#pragma unroll 8
        for (int j = 0; j < nb; ++j) {
            const unsigned short q0 = quant_u16(xs0[c0 + 2 * j], has_nd, nodata, scale, hi, nd);
            const unsigned short q1 = quant_u16(xs1[c0 + 2 * j], has_nd, nodata, scale, hi, nd);
            const unsigned int w = (unsigned int)(ok0 ? q0 : qfill) | ((unsigned int)(ok1 ? q1 : qfill) << 16);
            if (in0 && in1) *reinterpret_cast<unsigned int*>(o) = w;
            else if (in0) *o = (unsigned short)(w & 0xffffu);
            o += ostep;
        }
    }
    if (track) {
        // my pixels' bits over both band parities (lane ^ 16 holds the other half of my bands), then across the warps
        live0 &= __shfl_xor_sync(FULL, live0, 16);
        live1 &= __shfl_xor_sync(FULL, live1, 16);
        unsigned int w[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const unsigned int mine = hb == 0 ? ((((live0 >> r) & 1u) << (2 * pp)) | (((live1 >> r) & 1u) << (2 * pp + 1))) : 0u;
            w[r] = __reduce_or_sync(FULL, mine);
        }
        if (lane == 0) {
            hd->bk_word[stage][half][0] = w[0];
            hd->bk_word[stage][half][1] = w[1];
            hd->bk_word[stage][half][2] = w[2];
        }
        named_bar_sync(1 + stage, 32 * CPS);
        if (half == 0) {
            unsigned int a0 = 0xffffffffu, a1 = 0xffffffffu, a2 = 0xffffffffu;
#pragma unroll
            for (int c = 0; c < CPS; ++c) {
                a0 &= hd->bk_word[stage][c][0];
                a1 &= hd->bk_word[stage][c][1];
                a2 &= hd->bk_word[stage][c][2];
            }
            if (m != META_OOB) P.black[tile * TILE + lane] = (uint8_t)(((a0 | a1 | a2) >> lane) & 1u);
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(nthreads_of(MODE), 1) glt_stream_kernel(const StreamParams P) {
    constexpr int CPS = cps_of(MODE);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SmemHeader* hd = reinterpret_cast<SmemHeader*>(smem_raw);
    float* wt = reinterpret_cast<float*>(smem_raw + header_bytes());
    const int wt_bytes = (MODE & MODE_SRF) ? ((P.K * P.wt_pitch * 4 + 127) / 128 * 128) : 0;
    float4* stages = reinterpret_cast<float4*>(smem_raw + header_bytes() + wt_bytes);

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    const long long bid = blockIdx.x;
    const long long grid = gridDim.x;
    const int nstage = P.nstage;
    const int nprod = P.nprod;

    if (tid == 0) {
        for (int s = 0; s < MAX_STAGES; ++s) {
            mbar_init(&hd->full[s], 1);
            mbar_init(&hd->empty[s], CPS);
        }
        fence_mbar_init();
    }
    if ((MODE & MODE_SRF) && tid < P.K) hd->fill_out[tid] = P.fill_out ? P.fill_out[tid] : 0.f;
    {   // stale or uninitialised words in the gaps between runs would only cost the scan's slow path;
        // start from zeros so that behaviour does not depend on what the previous kernel left behind
        const int total = P.nstage * P.stage_f4;
        for (int i = tid; i < total; i += (int)blockDim.x) stages[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        fence_proxy_async_smem();  // the bulk copies (async proxy) overwrite these generic-proxy stores
    }
    __syncthreads();
    // From here the producers stream; the consumers build the SRF tables meanwhile (their first tile is ~2 us of GLT
    // and raw-cube latency away), synchronising among themselves on a named barrier.
    if ((MODE & MODE_SRF) && warp >= nprod) {
        const int ncons = (int)blockDim.x - 32 * nprod, ctid = tid - 32 * nprod, cwarp = warp - nprod;
        // transposed weight table Wt[k][b] = W[b][k], zero padded; W is read linearly (coalesced)
        const int total = P.bands * P.K;
        for (int i = ctid; i < total; i += ncons) {
            const int b = i / P.K, k = i - b * P.K;
            wt[k * P.wt_pitch + b] = P.W[i];
        }
        const int pad = P.wt_pitch - P.bands;
        for (int i = ctid; i < pad * P.K; i += ncons) wt[(i / pad) * P.wt_pitch + P.bands + i % pad] = 0.f;
        named_bar_sync(10, ncons);
        // contiguous non-zero run [first, last] of each folded response (one warp per band) ...
        for (int k = cwarp; k < P.K; k += (ncons >> 5)) {
            int first = 0x7fffffff, last = -1;
            for (int b = lane; b < P.bands; b += 32) {
                if (!(wt[k * P.wt_pitch + b] == 0.f)) {
                    first = first < b ? first : b;
                    last = b;
                }
            }
            first = __reduce_min_sync(0xffffffffu, first);
            last = __reduce_max_sync(0xffffffffu, last);
            if (lane == 0) {
                hd->krun[0][k] = last < 0 ? 0 : (first & ~3);
                hd->krun[1][k] = last < 0 ? 0 : last + 1;
            }
        }
        named_bar_sync(10, ncons);
        // ... then deal the bands to the CPS consumer warps of a stage: longest run first (ties: lowest band), to the
        // lighter warp.  One warp, lane = band, an arg-max reduction per pick.
        if (cwarp == 0) {
            const int len = lane < P.K ? hd->krun[1][lane] - hd->krun[0][lane] : -1;
            bool done = lane >= P.K;
            int load[CPS], cnt[CPS];
#pragma unroll
            for (int h = 0; h < CPS; ++h) load[h] = cnt[h] = 0;
            for (int n = 0; n < P.K; ++n) {
                const int key = done ? -1 : ((len << 5) | (31 - lane));
                const int top = __reduce_max_sync(0xffffffffu, key);
                const int best = 31 - (top & 31), bl = top >> 5;
                if (lane == best) done = true;
                const int b0 = hd->krun[0][best], b1 = hd->krun[1][best];
                int b1v = (b1 + 3) & ~3;
                if (b1v > (P.bands & ~3)) b1v = P.bands & ~3;
                if (b1v < b0) b1v = b0;
                int h = 0;
#pragma unroll
                for (int c = 1; c < CPS; ++c)
                    if (load[c] < load[h]) h = c;
#pragma unroll
                for (int c = 0; c < CPS; ++c)
                    if (c == h) {
                        if (lane == 0) hd->kparam[c][cnt[c]] = make_int4(best, b0, b1v, b1);
                        ++cnt[c];
                        load[c] += bl + 12;  // + fixed cost per band (loop set-up, store)
                    }
            }
            if (lane == 0) {
#pragma unroll
                for (int h = 0; h < CPS; ++h) hd->kcount[h] = cnt[h];
            }
        }
        named_bar_sync(10, ncons);
    }

    if (warp < nprod) {
        // =================================================================== PRODUCERS
        // Pixel and tile indices fit 32 bits (the ABI rejects grids of 2^31 pixels); only byte addresses are 64-bit.
        const unsigned int FULLM = 0xffffffffu;
        const int B = P.bands;
        const int npix = (int)P.npix, ntiles = (int)P.ntiles, igrid = (int)grid, ibid = (int)bid;
        const int raw_w = (int)P.raw_w, raw_h = (int)P.raw_h;
        const bool contiguous = P.glt_row_stride == P.out_w;
        const bool glt_ring = P.glt_ring && !P.identity;
        int(*gring)[2][TILE] = hd->glt[warp];
        auto tile_is_full = [&](int tile) { return tile * TILE + TILE <= npix; };
        // The 2 x 128 bytes of a tile's GLT entries are staged GLT_DEPTH tiles ahead: sixteen lanes issue one 16-byte
        // cp.async each and every lane commits one group per iteration (an empty one when nothing was issued), so "the
        // oldest group has landed" is cp.async.wait_group GLT_DEPTH - 1 — no mbarrier, no elected lane, no entry in the
        // SM's bulk-copy queue.  Faster than 1-D bulk copies into the same ring: all-nodata grid 0.107 -> 0.098 ms,
        // granule 0.3316 -> 0.3289 ms (profiles/r2/nodata/invalid_knobs_producer.log).
        auto issue_glt = [&](int g, int tile, bool on) {  // all lanes; on = warp-uniform "this tile's GLT is staged"
            if (on && lane < 16)
                glt_cp_async16(&gring[g][lane >> 3][(lane & 7) << 2],
                               (lane < 8 ? P.glt_x : P.glt_y) + (long long)tile * TILE + ((lane & 7) << 2));
            glt_cp_async_commit();
        };
        // A stage has ONE producer (a single waiter per `empty` barrier keeps the phase parity
        // unambiguous): this warp walks its stages w, w + nprod, ... round-robin; use `u` of stage
        // `s` is iteration u * nstage + s of the CTA, i.e. tile bid + (u * nstage + s) * grid.
        // Tiles are tracked as 64-bit only for the end test (the last step may pass 2^31).
        auto advance = [&](int& s, int& u) {
            s += nprod;
            if (s >= nstage) {
                s = warp;
                ++u;
            }
        };
        auto tile_of = [&](int s, int u) { return (long long)ibid + ((long long)u * nstage + s) * igrid; };
        int ps = warp, pu = 0;  // prefetch cursor of the GLT ring, GLT_DEPTH iterations ahead
        if (glt_ring) {
            for (int g = 0; g < GLT_DEPTH; ++g) {
                const long long tile = tile_of(ps, pu);
                issue_glt(g, (int)tile, tile < ntiles && tile_is_full((int)tile));
                advance(ps, pu);
            }
        }
        unsigned int cnt_nz = 0, cnt_ib = 0, cnt_ow = 0;
        // the raw cube is read once: evict-first keeps it from displacing the planes this kernel writes, which the
        // fit and apply kernels read next, from L2
        const uint64_t evict_first = l2_policy_evict_first();
        int stage = warp, use = 0;
        const bool pfill = producer_fills<MODE>(P);
        const bool fill_vec = pfill && (reinterpret_cast<uintptr_t>(P.bands_out) & 15) == 0 && (P.plane_stride & 3) == 0;
        unsigned int fills = 0;  // pfill: how often this producer has filled its (one) stage
        int g = 0;
        const unsigned int le = FULLM >> (31 - lane);  // lanes <= this one
        const int tbank = (P.bank_step * lane) & 31;
        if (warp < nstage)
        for (;;) {
            const long long tile64 = tile_of(stage, use);
            if (tile64 >= ntiles) break;
            const int tile = (int)tile64;
            const int p = tile * TILE + lane;
            const bool inb = p < npix;

            int gx = 0, gy = 0;
            if (!P.identity) {
                if (glt_ring) {
                    glt_cp_async_wait<GLT_DEPTH - 1>();   // my own copies of the oldest group ...
                    __syncwarp();                         // ... and every other lane's
                    if (tile_is_full(tile)) {
                        gx = gring[g][0][lane];
                        gy = gring[g][1][lane];
                        __syncwarp();
                    } else if (inb) {
                        gx = __ldg(P.glt_x + p);
                        gy = __ldg(P.glt_y + p);
                    }
                    const long long nt = tile_of(ps, pu);
                    issue_glt(g, (int)nt, nt < ntiles && tile_is_full((int)nt));
                    advance(ps, pu);
                    if (++g == GLT_DEPTH) g = 0;
                } else if (inb) {
                    const long long gi = contiguous ? (long long)p
                                                    : (long long)(p / (int)P.out_w) * P.glt_row_stride + (p % (int)P.out_w);
                    gx = __ldg(P.glt_x + gi);
                    gy = __ldg(P.glt_y + gi);
                }
            }
            // validity rule: emit_proj.py:691 (both != 0), :694 (1-based -> 0-based), :698-703 (in bounds).
            // (unsigned)(g - 1) < size is 0 <= g - 1 < size, and it is false for g = INT_MIN as well
            // (numpy's int32 g - 1 wraps to INT_MAX there, out of bounds too).
            const bool nz = (gx != 0) && (gy != 0);
            const unsigned int x0 = (unsigned int)gx - 1u, y0 = (unsigned int)gy - 1u;
            unsigned int lim_h = (unsigned int)raw_h, row_base = 0u;
            if (P.batch_out_rows) {  // tile batch: the entry indexes the raw tile of this ortho row's tile
                const unsigned int t = (unsigned int)(p / (int)P.out_w) / (unsigned int)P.batch_out_rows;
                lim_h = (unsigned int)P.batch_raw_rows;
                row_base = t * (unsigned int)P.batch_raw_rows;
            }
            bool ib = inb && nz && x0 < (unsigned int)raw_w && y0 < lim_h;  // the reference's valid_glt2
            // slow-axis index relative to the window held at P.raw (wraps to a huge value below the window)
            const unsigned int slow = (P.transpose ? x0 : y0 + row_base) - P.win_lo;
            const bool in_win = slow < P.win_n;
            int q = P.transpose ? (int)slow * raw_h + (int)y0 : (int)slow * raw_w + (int)x0;  // source pixel index
            if (P.identity) {
                ib = inb;
                q = p;
            }
            if (inb && !P.identity) {
                if (P.valid) P.valid[p] = ib ? 1 : 0;
                cnt_nz += nz ? 1u : 0u;
                cnt_ib += ib ? 1u : 0u;
                cnt_ow += (ib && !in_win) ? 1u : 0u;
            }
            if (!P.identity) ib = ib && in_win;  // a valid entry whose source row was not staged gets the fill value
                                                 // and is COUNTED (diag[3]): the host treats a non-zero count as an error
            if (!ib) q = 0;

            const unsigned int vmask = __ballot_sync(FULLM, ib);
            if (pfill && vmask == 0u && tile_is_full(tile)) {  // nodata tile: finished here, the ring never sees it
                if (fill_vec) {  // 8 lanes x 16 bytes cover a plane's 32 pixels: four planes per store instruction
                    for (int k = lane >> 3; k < P.K; k += 4) {
                        const float f = hd->fill_out[k];
                        *reinterpret_cast<float4*>(P.bands_out + (long long)k * P.plane_stride + (long long)tile * TILE +
                                                   ((lane & 7) << 2)) = make_float4(f, f, f, f);
                    }
                } else {
                    for (int k = 0; k < P.K; ++k) P.bands_out[(long long)k * P.plane_stride + p] = hd->fill_out[k];
                }
                if (P.fit_mask) P.fit_mask[p] = 0;
                advance(stage, use);
                continue;
            }
            // ---- runs: lane l continues lane l-1's run when its source pixel is the same or the next one
            const int qprev = __shfl_up_sync(FULLM, q, 1);
            const bool prev_ok = lane > 0 && ((vmask >> (lane - 1)) & 1u);
            const unsigned int dq = (unsigned int)(q - qprev);
            const bool cont = ib && prev_ok && P.merge && dq <= 1u;
            const bool head = ib && !cont;
            const unsigned int hmask = __ballot_sync(FULLM, head);
            const int hl = ib ? 31 - __clz((int)(hmask & le)) : lane;  // head lane of my run
            const unsigned int stops = (hmask | ~vmask) & ~le;         // first lane after my run (heads only)
            const int el = (stops ? __ffs((int)stops) - 1 : 32) - 1;   // last lane of the run I head
            const int q_head = __shfl_sync(FULLM, q, hl);
            const int q_last = __shfl_sync(FULLM, q, el);
            const int run_px = head ? q_last - q_head + 1 : 0;

            const float* src = P.raw + (long long)q * P.raw_pix_stride;  // heads: first spectrum of the run
            const unsigned long long a = reinterpret_cast<unsigned long long>(src);
            const unsigned long long lo = a & ~15ull;
            const int sp = (int)((a & 15ull) >> 2);
            const int run_words = sp + run_px * B;  // merge implies pixel stride == B
            const unsigned int bytes = head ? (unsigned int)((run_words + 3) >> 2) * 16u : 0u;
            // the 16-byte aligned window may stick out of the allocation by < 16 bytes at either end: those two
            // 16-byte pieces are then fetched word by word (only the words that belong to the cube)
            const bool clip_front = head && lo < P.raw_lo;
            const bool clip_back = head && lo + bytes > P.raw_hi;
            const unsigned int cut_front = clip_front ? 16u : 0u;
            const unsigned int cut = cut_front + (clip_back ? 16u : 0u);
            const unsigned int tma_bytes = bytes > cut ? bytes - cut : 0u;

            // ---- place the runs: each gets a 128-byte aligned slot and starts `toff` bytes into it, chosen so
            //      that lane l's spectrum begins (within 3 words) at shared-memory bank bank_step*l mod 32.  Lanes
            //      of a run are one spectrum (bands = 285 = 29 mod 32 words) apart, so the consumers'
            //      lane-per-pixel scalar loads of band b hit 32 different banks instead of colliding at random.
            //      One warp scan carries both sums (in 16-byte units): slots in the low half, TMA bytes in the high.
            const unsigned int toff = head ? (unsigned int)(((tbank - sp) & 31) & ~3) * 4u : 0u;
            const unsigned int slot = head ? ((bytes + toff + 127u) & ~127u) : 0u;
            const unsigned int mine = (slot >> 4) | ((tma_bytes >> 4) << 16);
            unsigned int incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int v = __shfl_up_sync(FULLM, incl, o);
                if (lane >= o) incl += v;
            }
            const unsigned int base = (((incl - mine) & 0xffffu) << 4) + toff;  // byte offset of my run's window
            const int start_word = (int)(base >> 2) + sp;                      // heads: word offset of the first spectrum
            const int head_word = __shfl_sync(FULLM, start_word, hl);
            const int off = head_word + (q - q_head) * B;
            const unsigned int totals = __shfl_sync(FULLM, incl, 31);
            const unsigned int tx = (totals >> 16) << 4;

            mbar_wait(&hd->empty[stage], ((pfill ? fills : (unsigned int)use) & 1u) ^ 1u);
            ++fills;

            hd->meta[stage][lane] = inb ? (ib ? off : META_FILL) : META_OOB;
            if (lane == 0) {
                hd->fill_f4[stage] = (int)(totals & 0xffffu);
                hd->tile_id[stage] = tile;
            }
            unsigned char* sbase = reinterpret_cast<unsigned char*>(stages + (long long)stage * P.stage_f4);
            if (clip_front | clip_back) {
                float* dst = reinterpret_cast<float*>(sbase + base) + sp;
                const int n = run_px * B;
                int front_end = clip_front ? (4 - sp < n ? 4 - sp : n) : 0;  // elements in the window's first 16 bytes
                int back_beg = clip_back ? (int)(bytes >> 2) - 4 - sp : n;     // ... and in its last 16 bytes
                if (tma_bytes == 0u) front_end = n;                            // nothing left for the bulk copy
                if (back_beg < front_end) back_beg = front_end;
                for (int i = 0; i < front_end; ++i) dst[i] = __ldg(src + i);
                for (int i = back_beg; i < n; ++i) dst[i] = __ldg(src + i);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_expect_tx(&hd->full[stage], tx);
            if (tma_bytes) {
                if (P.identity)  // un-fused SRF: no hint (its L2 behaviour with evict-first has not been measured)
                    bulk_g2s(sbase + base + cut_front, reinterpret_cast<const void*>(lo + cut_front), tma_bytes,
                             &hd->full[stage]);
                else
                    bulk_g2s_hint(sbase + base + cut_front, reinterpret_cast<const void*>(lo + cut_front), tma_bytes,
                                  &hd->full[stage], evict_first);
            }

            advance(stage, use);
        }
        if (pfill && warp < nstage) {  // end of this stage's sequence
            mbar_wait(&hd->empty[warp], (fills & 1u) ^ 1u);
            if (lane == 0) {
                hd->tile_id[warp] = -1;
                mbar_arrive_expect_tx(&hd->full[warp], 0u);
            }
        }
        if (P.diag && !P.identity) {
            const int snz = warp_sum((int)cnt_nz), sib = warp_sum((int)cnt_ib), sow = warp_sum((int)cnt_ow);
            if (lane == 0 && (snz | sib)) {
                atomicAdd(P.diag + 0, (unsigned long long)snz);
                atomicAdd(P.diag + 1, (unsigned long long)sib);
                atomicAdd(P.diag + 2, (unsigned long long)(snz - sib));
                if (P.has_view && sow) atomicAdd(P.diag + 3, (unsigned long long)sow);
            }
        }
    } else if (warp - nprod < CPS * nstage) {
        // =================================================================== CONSUMERS
        const int cw = warp - nprod;
        const int stage = cw / CPS;
        const int half = cw - stage * CPS;
        unsigned int use = 0;
        const float4* st4 = stages + (long long)stage * P.stage_f4;
        const long long tile_step = (long long)nstage * grid;
        const bool pfill = producer_fills<MODE>(P);
        for (long long tile = bid + (long long)stage * grid; pfill || tile < P.ntiles; tile += tile_step, ++use) {
            mbar_wait(&hd->full[stage], use & 1u);
            if (pfill) {
                tile = hd->tile_id[stage];
                if (tile < 0) break;
            }
            const int m = hd->meta[stage][lane];
            if (MODE & MODE_COPY) copy_tile<CPS>(P, st4, m, tile, lane, half);
            if (MODE & MODE_SRF) srf_tile<CPS>(P, hd, wt, st4, m, tile, lane, stage, half);
            if (MODE & MODE_Q16) {
                if (P.q16_pair) q16_tile2<CPS>(P, hd, st4, m, tile, lane, stage, half);
                else q16_tile<CPS>(P, hd, st4, m, tile, lane, stage, half);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&hd->empty[stage]);
        }
    }
}

// Fallback for short records (LOC / OBS planes, bands < 32): one thread per output element.
__global__ void __launch_bounds__(256) glt_small_kernel(const StreamParams P) {
    const long long total = P.npix * P.bands;
    unsigned int cnt_nz = 0, cnt_ib = 0, cnt_ow = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / P.bands;
        const int b = (int)(i - p * P.bands);
        const long long gi = (p / P.out_w) * P.glt_row_stride + (p % P.out_w);
        const int gx = __ldg(P.glt_x + gi), gy = __ldg(P.glt_y + gi);
        const bool nz = (gx != 0) && (gy != 0);
        const long long x0 = (long long)gx - 1, y0 = (long long)gy - 1;
        long long lim_h = P.raw_h, row_base = 0;
        if (P.batch_out_rows) {
            lim_h = P.batch_raw_rows;
            row_base = ((p / P.out_w) / P.batch_out_rows) * P.batch_raw_rows;
        }
        const bool ib = nz && x0 >= 0 && x0 < P.raw_w && y0 >= 0 && y0 < lim_h;
        const long long slow = (P.transpose ? x0 : y0 + row_base) - (long long)P.win_lo;
        const bool in_win = slow >= 0 && slow < (long long)P.win_n;
        float v = P.fill;
        if (ib && in_win) {
            const long long q = P.transpose ? slow * P.raw_h + y0 : slow * P.raw_w + x0;
            v = __ldg(P.raw + q * P.raw_pix_stride + b);
        }
        P.ortho[p * P.out_pix_stride + b] = v;
        if (b == 0) {
            if (P.valid) P.valid[p] = ib ? 1 : 0;
            cnt_nz += nz ? 1u : 0u;
            cnt_ib += ib ? 1u : 0u;
            cnt_ow += (ib && !in_win) ? 1u : 0u;
        }
    }
    if (P.diag) {
        const int snz = warp_sum((int)cnt_nz), sib = warp_sum((int)cnt_ib), sow = warp_sum((int)cnt_ow);
        if ((threadIdx.x & 31) == 0 && (snz | sib)) {
            atomicAdd(P.diag + 0, (unsigned long long)snz);
            atomicAdd(P.diag + 1, (unsigned long long)sib);
            atomicAdd(P.diag + 2, (unsigned long long)(snz - sib));
            if (P.has_view && sow) atomicAdd(P.diag + 3, (unsigned long long)sow);
        }
    }
}

// Slow-axis range (raw rows; raw columns when transposed) referenced by the valid, in-bounds entries of a GLT:
// range[0] = min, range[1] = max + 1 (caller initialises to {INT64_MAX, 0}); what a host stages for a mosaic slab or
// uploads for a granule (hsr_raw_view_t).  Same validity rule as the producers above.
__global__ void __launch_bounds__(256) glt_row_range_kernel(const int32_t* __restrict__ glt_x,
                                                            const int32_t* __restrict__ glt_y, long long n,
                                                            long long out_w, long long glt_row_stride,
                                                            unsigned int raw_h, unsigned int raw_w, int transpose,
                                                            unsigned long long* __restrict__ range) {
    unsigned int lo = 0xffffffffu, hi = 0u;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const long long gi = glt_row_stride == out_w ? p : (p / out_w) * glt_row_stride + (p % out_w);
        const int gx = __ldg(glt_x + gi), gy = __ldg(glt_y + gi);
        const unsigned int x0 = (unsigned int)gx - 1u, y0 = (unsigned int)gy - 1u;
        if (gx != 0 && gy != 0 && x0 < raw_w && y0 < raw_h) {
            const unsigned int slow = transpose ? x0 : y0;
            lo = slow < lo ? slow : lo;
            hi = slow + 1u > hi ? slow + 1u : hi;
        }
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0 && hi != 0u) {
        atomicMin(range + 0, (unsigned long long)lo);
        atomicMax(range + 1, (unsigned long long)hi);
    }
}

// ---------------------------------------------------------------------------- host side
// Run merging needs adjacent source pixels contiguous in memory (pixel stride == bands) and pays off only
// when spectra `bands` words apart fall into different banks (bands = 285: 29 mod 32, all 32 distinct).
bool merge_ok(int bands, long long pix_stride) {
    return pix_stride == bands && (bands & 3) != 0;
}

int plan_smem(StreamParams& P, int mode, size_t* smem_bytes) {
    // Stage capacity.  A run of n pixels is a 16-byte aligned window of 16 * ceil((3 + n * bands) / 4) bytes,
    // placed up to 112 bytes into a 128-byte aligned slot; a tile holds runs whose pixel counts sum to
    // <= TILE (un-merged: TILE runs of one pixel).  Worst case by a small knapsack over the run lengths.
    {
        long long f[TILE + 1], dp[TILE + 1];
        for (int n = 1; n <= TILE; ++n)
            f[n] = ((16LL * ((3 + (long long)n * P.bands + 3) / 4) + 112 + 127) / 128) * 128;
        dp[0] = 0;
        for (int t = 1; t <= TILE; ++t) {
            dp[t] = 0;
            const int nmax = P.merge ? t : 1;
            for (int n = 1; n <= nmax; ++n)
                if (f[n] + dp[t - n] > dp[t]) dp[t] = f[n] + dp[t - n];
        }
        P.stage_f4 = (int)((dp[TILE] + 128) / 16);  // + slack for the consumers' aligned 16-byte over-reads
    }
    // consecutive spectra of a run are `bands` words apart; runs of one pixel are spread with an odd step
    P.bank_step = P.merge ? (P.bands & 31) : 29;
    P.wt_pitch = (P.bands + 3) / 4 * 4;
    const size_t wt_bytes = (mode & MODE_SRF) ? ((size_t)P.K * P.wt_pitch * 4 + 127) / 128 * 128 : 0;
    const size_t fixed = (size_t)header_bytes() + wt_bytes;
    const size_t stage_bytes = (size_t)P.stage_f4 * 16;
    const size_t cap = (size_t)device_max_smem_optin();
    if (cap <= fixed + 128) return HSR_ENOSMEM;
    long long ns = (long long)((cap - fixed - 128) / stage_bytes);
    if (ns > MAX_STAGES) ns = MAX_STAGES;
    if (ns < 2) return HSR_ENOSMEM;
    P.nstage = (int)ns;
    P.nprod = P.nstage < MAX_PRODUCERS ? P.nstage : MAX_PRODUCERS;
    *smem_bytes = fixed + (size_t)P.nstage * stage_bytes;
    return HSR_OK;
}

template <int MODE>
int launch_stream(StreamParams& P, cudaStream_t stream) {
    size_t smem = 0;
    int rc = plan_smem(P, MODE, &smem);
    if (rc != HSR_OK) {
        set_error("spectrum of %d bands does not fit the shared-memory staging ring", P.bands);
        return rc;
    }
    static int smem_set[HSR_MAX_DEVICES];
    HSR_CUDA(ensure_dynamic_smem(glt_stream_kernel<MODE>, (int)smem, smem_set));
    long long grid = device_sm_count();
    if (grid > P.ntiles) grid = P.ntiles;
    glt_stream_kernel<MODE><<<(unsigned int)grid, 32 * (P.nprod + cps_of(MODE) * P.nstage), smem, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int check_view(const hsr_raw_view_t* v, long long raw_h, long long raw_w, int transpose, long long out_h) {
    if (!v) return HSR_OK;
    const long long slow_n = transpose ? raw_w : raw_h;
    HSR_REQUIRE(v->row0 >= 0 && v->rows >= 0 && v->row0 + v->rows <= slow_n, HSR_EINVAL,
                "raw view [%lld, %lld) outside the cube's %lld rows", (long long)v->row0, (long long)(v->row0 + v->rows), slow_n);
    HSR_REQUIRE(v->batch_out_rows >= 0 && v->batch_raw_rows >= 0 && (v->batch_out_rows > 0) == (v->batch_raw_rows > 0),
                HSR_EINVAL, "batch_out_rows / batch_raw_rows must both be positive or both be 0");
    if (v->batch_out_rows > 0) {
        HSR_REQUIRE(!transpose, HSR_EINVAL, "tile batches are not defined for transpose_raw_yx");
        HSR_REQUIRE(out_h % v->batch_out_rows == 0 && (out_h / v->batch_out_rows) * v->batch_raw_rows <= raw_h, HSR_EINVAL,
                    "tile batch: %lld ortho rows are not a whole number of %lld-row tiles with %lld raw rows each inside "
                    "raw_h = %lld", out_h, (long long)v->batch_out_rows, (long long)v->batch_raw_rows, raw_h);
    }
    return HSR_OK;
}

int check_common(const float* raw, long long raw_h, long long raw_w, int bands, long long raw_pix_stride,
                 const int32_t* glt_x, const int32_t* glt_y, long long out_h, long long out_w,
                 long long glt_row_stride) {
    HSR_REQUIRE(raw && glt_x && glt_y, HSR_EINVAL, "null raw / GLT pointer");
    HSR_REQUIRE(raw_h > 0 && raw_w > 0 && bands > 0, HSR_EINVAL, "raw shape must be positive (got %lld x %lld x %d)",
                raw_h, raw_w, bands);
    HSR_REQUIRE(out_h >= 0 && out_w >= 0, HSR_EINVAL, "negative ortho shape");
    HSR_REQUIRE(raw_h * raw_w < MAX_PIXELS && out_h * out_w < MAX_PIXELS, HSR_ERANGE,
                "raw and ortho grids are limited to 2^31 - 64 pixels each");
    HSR_REQUIRE(raw_pix_stride >= bands, HSR_EINVAL, "raw_pix_stride %lld < bands %d", raw_pix_stride, bands);
    HSR_REQUIRE(glt_row_stride >= out_w, HSR_EINVAL, "glt_row_stride %lld < out_w %lld", glt_row_stride, out_w);
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(raw) & 3) == 0, HSR_EALIGN, "raw is not 4-byte aligned");
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(glt_x) | reinterpret_cast<uintptr_t>(glt_y)) & 3) == 0, HSR_EALIGN,
                "GLT planes are not 4-byte aligned");
    return HSR_OK;
}

void fill_common(StreamParams& P, const float* raw, long long raw_h, long long raw_w, int bands,
                 long long raw_pix_stride, int transpose, const int32_t* glt_x, const int32_t* glt_y, long long out_h,
                 long long out_w, long long glt_row_stride, float fill, const hsr_raw_view_t* view) {
    P.raw = raw;
    P.raw_h = raw_h;
    P.raw_w = raw_w;
    P.raw_pix_stride = raw_pix_stride;
    P.bands = bands;
    P.transpose = transpose ? 1 : 0;
    P.identity = 0;
    P.merge = merge_ok(bands, raw_pix_stride) ? 1 : 0;
    P.glt_x = glt_x;
    P.glt_y = glt_y;
    P.out_w = out_w;
    P.glt_row_stride = glt_row_stride;
    P.npix = out_h * out_w;
    P.ntiles = (P.npix + TILE - 1) / TILE;
    P.glt_ring = (glt_row_stride == out_w || out_h <= 1) &&
                 ((reinterpret_cast<uintptr_t>(glt_x) | reinterpret_cast<uintptr_t>(glt_y)) & 15) == 0;
    P.fill = fill;
    const long long slow_n = transpose ? raw_w : raw_h, fast_n = transpose ? raw_h : raw_w;
    long long held = slow_n;
    P.win_lo = 0u;
    P.has_view = view ? 1 : 0;
    if (view && view->rows > 0) {
        P.win_lo = (unsigned int)view->row0;
        held = view->rows;
    }
    P.win_n = (unsigned int)held;
    P.batch_out_rows = view ? (int)view->batch_out_rows : 0;
    P.batch_raw_rows = view ? (int)view->batch_raw_rows : 0;
    P.raw_lo = reinterpret_cast<unsigned long long>(raw);
    P.raw_hi = P.raw_lo + ((unsigned long long)(held * fast_n - 1) * raw_pix_stride + bands) * 4ull;
}

}  // namespace

int glt_ortho_impl(const float* raw, long long raw_h, long long raw_w, int bands, long long raw_pix_stride,
                   int transpose, const int32_t* glt_x, const int32_t* glt_y, long long out_h, long long out_w,
                   long long glt_row_stride, float fill, float* out, long long out_pix_stride, uint8_t* valid,
                   unsigned long long* diag, const hsr_raw_view_t* view, cudaStream_t stream) {
    if (out_h == 0 || out_w == 0) return HSR_OK;  // empty grid: nothing to read or write
    int rc = check_common(raw, raw_h, raw_w, bands, raw_pix_stride, glt_x, glt_y, out_h, out_w, glt_row_stride);
    if (rc != HSR_OK) return rc;
    if ((rc = check_view(view, raw_h, raw_w, transpose, out_h)) != HSR_OK) return rc;
    HSR_REQUIRE(out, HSR_EINVAL, "null output pointer");
    HSR_REQUIRE(out_pix_stride >= bands, HSR_EINVAL, "out_pix_stride %lld < bands %d", out_pix_stride, bands);
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(out) & 3) == 0, HSR_EALIGN, "out is not 4-byte aligned");
    if (out_h == 0 || out_w == 0) return HSR_OK;
    StreamParams P{};
    fill_common(P, raw, raw_h, raw_w, bands, raw_pix_stride, transpose, glt_x, glt_y, out_h, out_w, glt_row_stride,
                fill, view);
    P.ortho = out;
    P.out_pix_stride = out_pix_stride;
    P.valid = valid;
    P.diag = diag;
    size_t smem = 0;
    if (bands >= 32 && plan_smem(P, MODE_COPY, &smem) == HSR_OK) return launch_stream<MODE_COPY>(P, stream);
    // short records: planes of the LOC / OBS cubes (emit_proj.py:1123-1131, :1217-1224)
    const long long total = P.npix * bands;
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)device_sm_count() * 16;
    if (blocks > cap) blocks = cap;
    glt_small_kernel<<<(unsigned int)blocks, 256, 0, stream>>>(P);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int glt_row_range_impl(const int32_t* glt_x, const int32_t* glt_y, long long out_h, long long out_w,
                       long long glt_row_stride, long long raw_h, long long raw_w, int transpose,
                       unsigned long long* range, cudaStream_t stream) {
    HSR_REQUIRE(glt_x && glt_y && range, HSR_EINVAL, "null GLT / range pointer");
    HSR_REQUIRE(out_h >= 0 && out_w >= 0 && glt_row_stride >= out_w, HSR_EINVAL, "bad GLT shape");
    HSR_REQUIRE(raw_h > 0 && raw_w > 0 && raw_h < MAX_PIXELS && raw_w < MAX_PIXELS, HSR_ERANGE, "bad raw shape");
    const long long n = out_h * out_w;
    if (n == 0) return HSR_OK;
    long long blocks = (n + 1023) / 1024;
    const long long cap = (long long)device_sm_count() * 8;
    if (blocks > cap) blocks = cap;
    glt_row_range_kernel<<<(unsigned int)blocks, 256, 0, stream>>>(glt_x, glt_y, n, out_w, glt_row_stride,
                                                                    (unsigned int)raw_h, (unsigned int)raw_w,
                                                                    transpose ? 1 : 0, range);
    HSR_CUDA(cudaGetLastError());
    return HSR_OK;
}

int glt_ortho_u16_impl(const float* raw, long long raw_h, long long raw_w, int bands, long long raw_pix_stride,
                       int transpose, const int32_t* glt_x, const int32_t* glt_y, long long out_h, long long out_w,
                       long long glt_row_stride, float fill, float scale, int has_nodata, float nodata, int nodata_u16,
                       uint16_t* out, long long plane_stride, uint8_t* valid, uint8_t* black, float nodata_tol,
                       float masked, float masked_tol, float zero_tol, unsigned long long* diag,
                       const hsr_raw_view_t* view, cudaStream_t stream) {
    if (out_h == 0 || out_w == 0) return HSR_OK;
    int rc = check_common(raw, raw_h, raw_w, bands, raw_pix_stride, glt_x, glt_y, out_h, out_w, glt_row_stride);
    if (rc != HSR_OK) return rc;
    if ((rc = check_view(view, raw_h, raw_w, transpose, out_h)) != HSR_OK) return rc;
    HSR_REQUIRE(out, HSR_EINVAL, "null output pointer");
    HSR_REQUIRE(plane_stride >= out_h * out_w, HSR_EINVAL, "plane_stride %lld < out_h*out_w", plane_stride);
    HSR_REQUIRE(nodata_u16 >= 1 && nodata_u16 <= 65535, HSR_ERANGE, "nodata_u16 = %d outside [1, 65535]", nodata_u16);
    HSR_REQUIRE((reinterpret_cast<uintptr_t>(out) & 1) == 0, HSR_EALIGN, "out is not 2-byte aligned");
    StreamParams P{};
    fill_common(P, raw, raw_h, raw_w, bands, raw_pix_stride, transpose, glt_x, glt_y, out_h, out_w, glt_row_stride,
                fill, view);
    P.valid = valid;
    P.diag = diag;
    P.q16 = out;
    P.q16_plane_stride = plane_stride;
    P.q16_pair = (reinterpret_cast<uintptr_t>(out) & 3) == 0 && (plane_stride & 1) == 0;
    P.q_scale = scale, P.q_nodata = nodata, P.q_hi = (float)(nodata_u16 - 1), P.q_has_nodata = has_nodata ? 1 : 0;
    P.q_nd = (unsigned short)nodata_u16;
    P.black = black;
    P.b_nodata_tol = nodata_tol, P.b_masked = masked, P.b_masked_tol = masked_tol, P.b_zero_tol = zero_tol;
    {   // what an invalid GLT pixel (every band == fill) turns into: same arithmetic as the device code, on the host
        const bool finite = fill == fill && fill - fill == 0.f;
        const bool vld = finite && !(has_nodata && fill == nodata);
        const float r = fill * scale;
        float t = r < 0.f ? 0.f : r;
        t = t > P.q_hi ? P.q_hi : t;
        unsigned int q = (unsigned int)__builtin_rintf(t);
        if (!(__builtin_fabsf(r) < 2147483648.f)) q = 0u;
        P.q_fill = vld ? (unsigned short)q : P.q_nd;
        auto close = [](float x, float y, float tol) { return __builtin_fabsf(x - y) <= tol || x == y; };
        P.black_fill = ((has_nodata && close(fill, nodata, nodata_tol)) ? 1 : 0) | (close(fill, masked, masked_tol) ? 2 : 0) |
                       ((__builtin_fabsf(fill) < zero_tol) ? 4 : 0);
    }
    size_t smem = 0;
    HSR_REQUIRE(bands >= 32 && plan_smem(P, MODE_Q16, &smem) == HSR_OK, HSR_ERANGE,
                "hsr_glt_ortho_u16 needs 32 <= bands and a spectrum that fits the staging ring (got %d)", bands);
    return launch_stream<MODE_Q16>(P, stream);
}

int glt_srf_impl(const float* raw, long long raw_h, long long raw_w, int bands, long long raw_pix_stride,
                 int transpose, const int32_t* glt_x, const int32_t* glt_y, long long out_h, long long out_w,
                 long long glt_row_stride, float fill, const float* W, const float* fill_out, int K,
                 float* bands_out, long long bands_plane_stride, float* ortho_out, long long out_pix_stride,
                 uint8_t* valid, unsigned long long* diag, uint8_t* fit_mask, int gate_k, float gate_gt,
                 const hsr_raw_view_t* view, cudaStream_t stream) {
    if (out_h == 0 || out_w == 0) return HSR_OK;
    int rc = check_common(raw, raw_h, raw_w, bands, raw_pix_stride, glt_x, glt_y, out_h, out_w, glt_row_stride);
    if (rc != HSR_OK) return rc;
    if ((rc = check_view(view, raw_h, raw_w, transpose, out_h)) != HSR_OK) return rc;
    HSR_REQUIRE(W && fill_out && bands_out, HSR_EINVAL, "null W / fill_out / bands_out pointer");
    HSR_REQUIRE(K >= 1 && K <= MAXK, HSR_ERANGE, "K = %d outside [1, %d]", K, MAXK);
    HSR_REQUIRE(gate_k < K, HSR_EINVAL, "gate_k = %d >= K = %d", gate_k, K);
    HSR_REQUIRE(bands_plane_stride >= out_h * out_w, HSR_EINVAL, "bands_plane_stride %lld < out_h*out_w",
                bands_plane_stride);
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(bands_out)) & 3) == 0, HSR_EALIGN,
                "W / bands_out not 4-byte aligned");
    if (ortho_out) {
        HSR_REQUIRE(out_pix_stride >= bands, HSR_EINVAL, "out_pix_stride %lld < bands %d", out_pix_stride, bands);
        HSR_REQUIRE((reinterpret_cast<uintptr_t>(ortho_out) & 3) == 0, HSR_EALIGN, "ortho_out not 4-byte aligned");
    }
    if (out_h == 0 || out_w == 0) return HSR_OK;
    StreamParams P{};
    fill_common(P, raw, raw_h, raw_w, bands, raw_pix_stride, transpose, glt_x, glt_y, out_h, out_w, glt_row_stride,
                fill, view);
    P.W = W;
    P.fill_out = fill_out;
    P.K = K;
    P.bands_out = bands_out;
    P.plane_stride = bands_plane_stride;
    P.ortho = ortho_out;
    P.out_pix_stride = out_pix_stride;
    P.valid = valid;
    P.diag = diag;
    P.fit_mask = fit_mask;
    P.gate_k = fit_mask ? gate_k : -1;
    P.gate_gt = gate_gt;
    if (ortho_out) return launch_stream<MODE_COPY | MODE_SRF>(P, stream);
    return launch_stream<MODE_SRF>(P, stream);
}

int srf_impl(const float* cube, long long n_pix, int bands, long long pix_stride, const float* W, int K,
             float* bands_out, long long bands_plane_stride, uint8_t* fit_mask, int gate_k, float gate_gt,
             cudaStream_t stream) {
    HSR_REQUIRE(cube && W && bands_out, HSR_EINVAL, "null cube / W / bands_out pointer");
    HSR_REQUIRE(n_pix >= 0 && bands > 0, HSR_EINVAL, "bad cube shape (%lld x %d)", n_pix, bands);
    HSR_REQUIRE(n_pix < MAX_PIXELS, HSR_ERANGE, "cubes are limited to 2^31 - 64 pixels");
    HSR_REQUIRE(pix_stride >= bands, HSR_EINVAL, "pix_stride %lld < bands %d", pix_stride, bands);
    HSR_REQUIRE(K >= 1 && K <= MAXK, HSR_ERANGE, "K = %d outside [1, %d]", K, MAXK);
    HSR_REQUIRE(bands_plane_stride >= n_pix, HSR_EINVAL, "bands_plane_stride %lld < n_pix", bands_plane_stride);
    HSR_REQUIRE(((reinterpret_cast<uintptr_t>(cube) | reinterpret_cast<uintptr_t>(W) |
                  reinterpret_cast<uintptr_t>(bands_out)) & 3) == 0,
                HSR_EALIGN, "cube / W / bands_out not 4-byte aligned");
    if (n_pix == 0) return HSR_OK;
    StreamParams P{};
    P.raw = cube;
    P.raw_h = 1;
    P.raw_w = n_pix;
    P.raw_pix_stride = pix_stride;
    P.bands = bands;
    P.identity = 1;
    P.win_lo = 0u;
    P.win_n = 1u;
    P.merge = merge_ok(bands, pix_stride) ? 1 : 0;
    P.out_w = n_pix;
    P.glt_row_stride = n_pix;
    P.npix = n_pix;
    P.ntiles = (n_pix + TILE - 1) / TILE;
    P.raw_lo = reinterpret_cast<unsigned long long>(cube);
    P.raw_hi = P.raw_lo + ((unsigned long long)(n_pix - 1) * pix_stride + bands) * 4ull;
    P.W = W;
    P.K = K;
    P.bands_out = bands_out;
    P.plane_stride = bands_plane_stride;
    HSR_REQUIRE(gate_k < K, HSR_EINVAL, "gate_k = %d >= K = %d", gate_k, K);
    P.fit_mask = fit_mask;
    P.gate_k = fit_mask ? gate_k : -1;
    P.gate_gt = gate_gt;
    return launch_stream<MODE_SRF>(P, stream);
}

}  // namespace hsr
