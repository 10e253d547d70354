/*
 * hsr_b200.h — C ABI of libhsr_b200.so: the EMIT -> Sentinel-2 pair-synthesis hot path
 * (GLT orthorectification, SRF band synthesis, per-band polynomial colour matching)
 * as hand-written sm_100a CUDA kernels.
 *
 * The reference (martasumyk/hyperspectral_super-resolution) has no FFI of its own: its
 * boundary is the Python call surface of EMIT_data/emit_proj.py, s2_emit/srf.py,
 * s2_emit/synth.py and s2_emit/poly_regression.py.  Each entry point below names the
 * reference lines whose arithmetic it replaces; INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (a torch.Tensor's data_ptr());
 *     the library allocates nothing and keeps no global state, so calls are re-entrant
 *     across streams and threads;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 = OK, < 0 = HSR_E* argument error, > 0 = cudaError_t;
 *     hsr_last_error() returns a thread-local message for the last non-zero return;
 *   - strides are in ELEMENTS, not bytes.
 */
#ifndef HSR_B200_H
#define HSR_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define HSR_API __attribute__((visibility("default")))
#else
#define HSR_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define HSR_ABI_VERSION 7

enum {
    HSR_OK = 0,
    HSR_EINVAL = -1,    /* bad size / null pointer / negative stride */
    HSR_EALIGN = -2,    /* pointer not 4-byte aligned, or output not 16-byte aligned */
    HSR_ERANGE = -3,    /* bands / K / deg outside the supported range */
    HSR_ENOSMEM = -4,   /* spectrum too long for the shared-memory staging ring */
    HSR_EPEER = -5,     /* hsr_peer_status: a peer exchange timed out (see HSR_PEER_TIMEOUT) */
    HSR_ENCCL = -6      /* hsr_allreduce_moments: NCCL not loadable, or ncclAllReduce failed */
};

/* limits (compile-time constants of the kernels) */
#define HSR_MAX_SRF_BANDS 16     /* K: synthesised S2 bands per launch            */
#define HSR_MAX_POLY_DEG 8       /* polynomial degree                             */
#define HSR_TILE_PX 32           /* ortho pixels per staged tile                  */
#define HSR_MAX_PERCENTILES 2    /* percentiles per hsr_masked_percentiles_f64 call (pmin, pmax) */

/* flags of hsr_fit_moments_f64 */
#define HSR_FIT_MASK_GIVEN 1     /* `valid` already IS the fit mask: use it as given, write no mask   */
#define HSR_FIT_Y_FINITE 2       /* the computed mask also requires every y[k] to be finite            */

/* cross-GPU exchange of the fit moments over NVLink peer memory */
#define HSR_PEER_MAX_RANKS 16
#define HSR_PEER_MAX_DOUBLES 1024    /* moments per rank and exchange: K * G * (3*deg+2) */
#define HSR_IPC_HANDLE_BYTES 64
#define HSR_PEER_DEFAULT_TIMEOUT_MS 10000u  /* hsr_exchange_t.timeout_ms == 0 */
#define HSR_PEER_TIMEOUT 1u                 /* status bit of hsr_peer_status */

/*
 * One exchange = "sum the K*G*(3*deg+2) moments over all ranks", fused into the two kernels either side of it
 * instead of a collective call: hsr_fit_moments_f64 stores this rank's sums into every rank's peer block (remote
 * stores over NVLink / NVSwitch) and raises a flag there; hsr_poly_solve_apply_f32 polls its own block until all
 * flags carry the epoch and adds the slots in rank order (bit-identical on every rank).  Pass the SAME struct to
 * both calls; NULL or nranks <= 1 = single GPU.
 *   peer_blocks   DEVICE array [nranks] of device pointers: every rank's peer block as mapped into THIS process
 *                 (own block: hsr_peer_alloc; the others: hsr_ipc_import of the handles the peers exported).
 *   epoch         0: the kernels number the exchanges themselves (a counter in the peer block; every rank must take
 *                 part in every exchange) — nothing in the arguments changes from call to call, so the step can be
 *                 replayed from a CUDA graph; or 1, 2, 3, ... given by the host, the same on every rank.
 *   timeout_ms    how long a block of hsr_poly_solve_apply_f32 polls for the peers' flags (0 = the default,
 *                 HSR_PEER_DEFAULT_TIMEOUT_MS).  The wait is BOUNDED: if a peer never publishes this epoch (it died,
 *                 raised before its fit, or the ranks ran different numbers of exchanges) the kernel gives up, writes
 *                 NaN coefficients (never a silent per-rank fit) and sets HSR_PEER_TIMEOUT in the block's sticky
 *                 status word; hsr_peer_status returns HSR_EPEER from then on.
 * Contract: on one stream, calls with an exchange strictly alternate fit, solve/apply, fit, ... and every rank
 * performs the same number of exchanges.
 */
typedef struct hsr_exchange {
    void* const* peer_blocks;
    void* my_block;
    int nranks;
    int rank;
    unsigned long long epoch;
    unsigned int timeout_ms;
    unsigned int reserved;
} hsr_exchange_t;

/*
 * Optional view of the raw cube for the three GLT entry points (NULL = the whole cube is at `raw`, one granule):
 *   row0, rows     `raw` points at slow-axis index row0 and holds `rows` of them (raw rows; raw columns when
 *                  transpose_raw_yx) — rows == 0 means all.  raw_h / raw_w stay the LOGICAL size of the cube, so the
 *                  validity rule (emit_proj.py:698-703), `valid` and diag[0..2] do not change.  For mosaic slabs whose
 *                  GLT references a band of the raw mosaic (stage only min..max gy of the slab, SURVEY 7.3-6) and for
 *                  hosts that upload only the rows a granule's GLT touches.  A valid entry whose source lies outside the
 *                  window gets the fill value and is counted in diag[3]: the caller must treat a non-zero count as an
 *                  error (it sized the window wrongly).
 *   batch_out_rows, batch_raw_rows   both > 0: the ortho grid is a stack of out_h / batch_out_rows independent tiles
 *                  (tiles_helpers' batch, tiles_helpers/utils.py:256-277); the GLT entries of tile t are 1-based indices
 *                  into ITS raw tile, raw rows [t*batch_raw_rows, (t+1)*batch_raw_rows) of `raw`, and are in bounds iff
 *                  gy - 1 < batch_raw_rows (an entry pointing past its own tile is dropped, never read from a
 *                  neighbour).  Not defined for transpose_raw_yx.
 * With a view, diag is [4] u64.
 */
typedef struct hsr_raw_view {
    int64_t row0;
    int64_t rows;
    int64_t batch_out_rows;
    int64_t batch_raw_rows;
} hsr_raw_view_t;

/* workspace selectors for hsr_workspace_bytes */
enum { HSR_OP_POLY_MOMENTS = 1 };

HSR_API int hsr_version(void);
HSR_API const char* hsr_last_error(void);

/*
 * GLT orthorectification gather (bit-exact copy / fill).
 * Replaces EMIT_data/emit_proj.py:682-703 (GLT -> validity, 1-based -> 0-based, in-bounds
 * test), :947-948 (index lists), :968-987 (fill with -9999 then out[valid] = raw[gy, gx, :]),
 * and, with bands == 1, the plane gathers at :1123-1131 (LOC) and :1217-1224 (OBS);
 * equal to EMIT_data/emit_tools.py:153-181 (apply_glt) on in-range GLTs.
 *
 *   raw            [raw_h, raw_w, bands] f32, pixel stride raw_pix_stride (>= bands) elements;
 *                  if transpose_raw_yx != 0 the memory is [raw_w, raw_h, bands]
 *                  (dims (crosstrack, downtrack), emit_proj.py:646-661,976-977) and raw_h/raw_w
 *                  are the logical (downtrack, crosstrack) sizes.
 *   glt_x, glt_y   [out_h, out_w] int32 planes, row stride glt_row_stride; 1-based, 0 = nodata.
 *   out            [out_h, out_w, bands] f32, pixel stride out_pix_stride; rows are dense
 *                  (row stride = out_w * out_pix_stride).
 *   valid          nullable [out_h, out_w] u8: 1 where the GLT entry is non-zero AND in bounds.
 *   diag           nullable [3] u64 ([4] with a view), ACCUMULATED (caller zeroes): {valid_glt_count,
 *                  valid_glt_inbounds_count, valid_glt_dropped_oob} (emit_proj.py:705-718) [, outside_view].
 *   view           nullable hsr_raw_view_t (host memory, read during the call).
 */
HSR_API int hsr_glt_ortho_f32(const float* raw, int64_t raw_h, int64_t raw_w, int bands, int64_t raw_pix_stride,
                      int transpose_raw_yx, const int32_t* glt_x, const int32_t* glt_y,
                      int64_t out_h, int64_t out_w, int64_t glt_row_stride, float fill,
                      float* out, int64_t out_pix_stride, uint8_t* valid,
                      unsigned long long* diag, const hsr_raw_view_t* view, void* stream);

/*
 * Fused GLT gather + SRF band integration: the raw cube is read from HBM once.
 * Replaces the gather above followed by s2_emit/synth.py:32-43
 * (rsp = interp(..)*good; num = trapz(R*rsp); den = trapz(rsp); num/(den+1e-32)) with the
 * trapezoid rule and the normalisation folded on the host into W (see srf_fold_weights):
 *     bands_out[k, p] = sum_b raw[gy, gx, b] * W[b, k]          (fp32 FMA)
 * Invalid GLT pixels give fill_out[k] (= fill * sum_b W[b,k], host-precomputed) and valid = 0.
 * Non-finite samples propagate exactly as the dense product of synth.py:41 does: a NaN in ANY of
 * the `bands` samples, or an Inf under a zero weight (0 * Inf), gives NaN; an Inf under a
 * non-zero weight gives +-Inf.
 *
 *   W              [bands, K] f32 row-major.
 *   bands_out      [K, out_h*out_w] f32 planes, plane stride bands_plane_stride (>= out_h*out_w).
 *   ortho_out      nullable: also materialise the ortho cube exactly as hsr_glt_ortho_f32 does.
 *   fit_mask       nullable [out_h, out_w] u8 out: the fit mask of s2_emit/poly_regression.py:106 computed from
 *                  the planes as they are written — valid & all_k isfinite(bands_out[k]) &
 *                  (bands_out[gate_k] > gate_gt); gate_k < 0 disables the gate.  Identical to running
 *                  hsr_fit_mask_u8 on bands_out afterwards, without re-reading the planes.
 */
HSR_API int hsr_glt_srf_f32(const float* raw, int64_t raw_h, int64_t raw_w, int bands, int64_t raw_pix_stride,
                    int transpose_raw_yx, const int32_t* glt_x, const int32_t* glt_y,
                    int64_t out_h, int64_t out_w, int64_t glt_row_stride, float fill,
                    const float* W, const float* fill_out, int K,
                    float* bands_out, int64_t bands_plane_stride,
                    float* ortho_out, int64_t out_pix_stride, uint8_t* valid,
                    unsigned long long* diag, uint8_t* fit_mask, int gate_k, float gate_gt,
                    const hsr_raw_view_t* view, void* stream);

/*
 * Slow-axis range of the raw cube that a GLT (or a row slab of one) references: over the entries that pass the
 * validity rule of emit_proj.py:691-703, range[0] = min(gy - 1), range[1] = max(gy - 1) + 1 (gx when
 * transpose_raw_yx).  ACCUMULATED with min / max: the caller initialises range to {UINT64_MAX, 0}; an untouched
 * range means no valid entry.  What a host needs to size an hsr_raw_view_t (SURVEY 7.3-6: "stage only the raw rows a
 * slab references").
 */
HSR_API int hsr_glt_row_range(const int32_t* glt_x, const int32_t* glt_y, int64_t out_h, int64_t out_w,
                      int64_t glt_row_stride, int64_t raw_h, int64_t raw_w, int transpose_raw_yx,
                      unsigned long long* range /*[2] u64*/, void* stream);

/*
 * Un-fused SRF integration of an already orthorectified cube (the shape
 * s2_emit/synth.py:9-45 pseudo_s2_srf_integral is called with).
 *   cube           [n_pix, bands] f32, pixel stride pix_stride.
 *   bands_out      [K, n_pix] f32 planes, plane stride bands_plane_stride.
 *   fit_mask       nullable [n_pix] u8 out, as in hsr_glt_srf_f32 (every pixel counts as valid).
 */
HSR_API int hsr_srf_f32(const float* cube, int64_t n_pix, int bands, int64_t pix_stride,
                const float* W, int K, float* bands_out, int64_t bands_plane_stride,
                uint8_t* fit_mask, int gate_k, float gate_gt, void* stream);

/*
 * Polynomial regression, stage 1: fp64 moments of the normal equations, reduced
 * block -> grid in a fixed order (deterministic).  Replaces the Vandermonde/lstsq inside
 * np.polyfit as called at s2_emit/poly_regression.py:58-60 (and the pixel-paired per-band
 * fit of Pairs_EMIT_S2_demo-2.ipynb cell 72).
 *   x, y           K series of n f32 samples: element (k, i) at x[k*x_k_stride + i*x_n_stride].
 *   mask           nullable u8, rows of n; sample (k, i) is used iff
 *                  mask[((k / mask_k_div) % mask_k_mod)*n + i] != 0 AND x, y are finite
 *                  (poly_regression.py:35-36).  One shared mask: div = 1, mod = 1; one mask per
 *                  series: div = 1, mod = K; series laid out [band][tile] with one mask per tile:
 *                  div = 1, mod = n_tiles.
 *   moments        [K, 3*deg+2] f64: S_j = sum x^j (j = 0..2deg; S_0 = count) then
 *                  T_j = sum x^j y (j = 0..deg).
 *   partial        workspace of hsr_workspace_bytes(HSR_OP_POLY_MOMENTS, n, K, deg) bytes.
 */
HSR_API int hsr_poly_moments_f64(const float* x, int64_t x_k_stride, int64_t x_n_stride,
                         const float* y, int64_t y_k_stride, int64_t y_n_stride,
                         const uint8_t* mask, int64_t mask_k_div, int64_t mask_k_mod, int64_t n, int K,
                         int deg, double* partial, double* moments, void* stream);

/*
 * Stage 2: one warp per series solves the column-scaled normal equations in fp64.
 *   coeffs         [K, deg+1] f64, highest power first (np.polyfit order).
 *   min_count      series with S_0 < min_count get the identity polynomial
 *                  (coeffs[:, -2] = 1; poly_regression.py:38-41).
 */
HSR_API int hsr_poly_solve_f64(const double* moments, int K, int deg, int64_t min_count,
                       double* coeffs, void* stream);

/*
 * Stage 3: apply.  Replaces s2_emit/poly_regression.py:65-84 (apply_poly_rgb):
 * out = x; where mask: out = (f32) polyval_f64(coeffs[k], x); then EVERY sample is clipped
 * to [lo, hi] (NaN stays NaN).  Pass lo > hi to disable the clip.
 */
HSR_API int hsr_poly_apply_f32(const float* x, int64_t x_k_stride, int64_t x_n_stride,
                       const double* coeffs, const uint8_t* mask, int64_t mask_k_div, int64_t mask_k_mod,
                       int64_t n, int K, int deg, float lo, float hi,
                       float* out, int64_t out_k_stride, int64_t out_n_stride, void* stream);

/*
 * Fit mask of the pair-synthesis script, s2_emit/poly_regression.py:106 (and :118 when y is given):
 * mask[g, i] = valid[g, i] (if given) AND all_k isfinite(x[k, g, i]) AND x[gate_k, g, i] > gate_gt
 *              [AND all_k isfinite(y[k, g, i])].
 * x, y: element (k, g, i) at x[k*x_k_stride + g*x_g_stride + i]; y nullable; gate_k < 0 disables the gate.
 * (hsr_glt_srf_f32 can emit the same mask for free while it writes the planes.)
 */
HSR_API int hsr_fit_mask_u8(const float* x, int64_t x_k_stride, int64_t x_g_stride,
                    const float* y, int64_t y_k_stride, int64_t y_g_stride, int64_t n, int K, int G,
                    const uint8_t* valid, int gate_k, float gate_gt, uint8_t* mask, void* stream);

/*
 * Fit of the pair-synthesis pass: fit mask (hsr_fit_mask_u8, unless it is given) followed by the fp64 moments of
 * the K*G series (s2_emit/poly_regression.py:106 for the mask, :35-36 and :58-60 for the fit).
 *   x, y           K bands x G groups x n samples: element (k, g, i) at x[k*x_k_stride + g*x_g_stride + i]
 *                  (a granule: G = 1; a tile batch with one fit per tile: G = tiles, n = pixels per tile).
 *   valid          nullable [G, n] u8 (the GLT mask); gate_k < 0 disables the gate.
 *   mask           [G, n] u8 out: valid & all_k isfinite(x[k]) & (x[gate_k] > gate_gt); required unless
 *                  HSR_FIT_MASK_GIVEN.
 *   moments        [K, G, 3*deg+2] f64 over the samples with mask & isfinite(x[k]) & isfinite(y[k]); same layout
 *                  and meaning as hsr_poly_moments_f64 with K*G series (series s = k*G + g).
 *   flags          HSR_FIT_MASK_GIVEN: `valid` is the finished fit mask (e.g. of hsr_fit_mask_u8), nothing is
 *                  recomputed and `mask` is not written; HSR_FIT_Y_FINITE: the computed mask also needs every
 *                  y[k] finite (`valid60 &= isfinite(s2_real_60m).all(0)`, poly_regression.py:118).
 *   x_stretch, y_stretch   nullable [K*G][2] f64 (lo, hi) per series s = k*G + g: the samples enter the fit
 *                  as (f32) clip((f64(v) - lo) / (hi - lo + 1e-12), 0, 1) — the shared percentile stretch of
 *                  s2_emit/color.py:25-34 applied at poly_regression.py:126-127, never materialised.
 *   partial        workspace of hsr_fit_moments_workspace_bytes(n, K, G, deg) bytes.
 * K*G <= 65535.  Deterministic (fixed reduction order).
 */
HSR_API int hsr_fit_moments_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride,
                        const float* y, int64_t y_k_stride, int64_t y_g_stride,
                        const uint8_t* valid, int64_t n, int K, int G, int deg, int gate_k, float gate_gt,
                        int flags, const double* x_stretch, const double* y_stretch,
                        uint8_t* mask, double* partial, double* moments, const hsr_exchange_t* exchange,
                        void* stream);

HSR_API size_t hsr_fit_moments_workspace_bytes(int64_t n, int K, int G, int deg);

/*
 * Fused solve + apply (hsr_poly_solve_f64 followed by hsr_poly_apply_f32 in one launch): every block
 * re-solves its series' (deg+1) x (deg+1) system, then maps its share of the samples.
 *   moments        [K*G, 3*deg+2] f64 (after any cross-rank all-reduce).
 *   mask           nullable [G, n] u8, shared by the K bands of a group.
 *   x_stretch      nullable [K*G][2] f64 (lo, hi): x is percentile-stretched first (see hsr_fit_moments_f64).
 *   exchange       nullable: with nranks > 1 the system solved is the rank-ordered SUM of every rank's moments of
 *                  this epoch (see hsr_exchange_t; `moments` is then not read) — the all-reduce of the global fit,
 *                  done in this kernel's prologue; moments_out (nullable [K*G, 3*deg+2]) receives the sums.
 *   coeffs         [K*G, deg+1] f64 out, highest power first.
 *   out            element (k, g, i) at out[k*out_k_stride + g*out_g_stride + i].
 */
HSR_API int hsr_poly_solve_apply_f32(const float* x, int64_t x_k_stride, int64_t x_g_stride,
                             const double* moments, const uint8_t* mask, int64_t n, int K, int G, int deg,
                             int64_t min_count, float lo, float hi, const double* x_stretch, double* coeffs,
                             float* out, int64_t out_k_stride, int64_t out_g_stride,
                             const hsr_exchange_t* exchange, double* moments_out, void* stream);

/*
 * Local sum of a global fit over several units per rank (BASELINE configs[3]: 64 granules dealt to the ranks, ONE
 * fit): out[j] = sum over u of per_unit[u*count + j], u ascending (bit-reproducible), count = K*G*(3*deg+2).
 * With an exchange the sums are also published to every rank's peer block exactly as hsr_fit_moments_f64 would
 * (this call then takes the "fit" turn of the exchange; hsr_poly_solve_apply_f32 of the first unit consumes it and
 * its moments_out serves the remaining units).  units == 0 publishes zeros (a rank that was dealt nothing still takes
 * part in the exchange).
 */
HSR_API int hsr_moments_sum_f64(const double* per_unit, int units, int64_t count, double* out,
                        const hsr_exchange_t* exchange, void* stream);

HSR_API size_t hsr_workspace_bytes(int op, int64_t n, int K, int deg);

/*
 * Shared percentile stretch, s2_emit/color.py:25-34 (apply_shared_percentile_stretch; called between the SRF
 * synthesis and the fit at s2_emit/poly_regression.py:126-127).
 *
 * hsr_masked_percentiles_f64: out[s, j] = np.percentile(x[s][mask], 100*q[j]) for every series s = k*G + g
 * (element (k, g, i) at x[k*x_k_stride + g*x_g_stride + i], mask row g of n bytes, nullable = all samples),
 * EXACT: three launches and ONE pass over the planes — brackets from a sample, a streaming pass that counts what
 * lies below / at the bracket keys and collects what lies inside, a per-series finish (radix select among the
 * collected keys; over the whole series if a bracket missed) — and the interpolation follows numpy's
 * "linear" method operation by operation (float32 neighbour difference, float64 lerp, the gamma >= 0.5
 * branch), so results are bit-identical to numpy's float64 output.  A NaN among the masked samples, or no
 * masked sample at all, gives NaN (numpy raises IndexError for the empty case; the host wrapper mirrors that).
 *   q              [Q] f64 on the device, fractions in [0, 1] (percent / 100), Q <= HSR_MAX_PERCENTILES.
 *   workspace      hsr_percentiles_workspace_bytes(n, K, G, nsets) bytes, 256-byte aligned (nsets = 1; 2 for the pair).
 * n < 2^32 (the candidate and histogram counters are 32-bit), K*G <= 32767.
 * hsr_masked_percentiles_pair_f64: the same for TWO plane sets of one shape under one mask — the two images of the
 * stretch (poly_regression.py:126-127) — in the same three launches; out_x, out_y [K*G, Q].
 *
 * hsr_stretch_f32: out = (f32) clip((f64(x) - lo) / (hi - lo + 1e-12), 0, 1) with (lo, hi) = lohi[s] — the
 * float64 expression of color.py:33 stored as float32, bit-exact.  (hsr_fit_moments_f64 and
 * hsr_poly_solve_apply_f32 take the same [S][2] table and apply the stretch on the fly instead.)
 */
HSR_API size_t hsr_percentiles_workspace_bytes(int64_t n, int K, int G, int nsets);
HSR_API int hsr_masked_percentiles_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride, const uint8_t* mask,
                               int64_t n, int K, int G, const double* q, int Q, void* workspace,
                               double* out, void* stream);
HSR_API int hsr_masked_percentiles_pair_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride,
                                    const float* y, int64_t y_k_stride, int64_t y_g_stride, const uint8_t* mask,
                                    int64_t n, int K, int G, const double* q, int Q, void* workspace,
                                    double* out_x, double* out_y, void* stream);
HSR_API int hsr_stretch_f32(const float* x, int64_t x_k_stride, int64_t x_g_stride, const double* lohi,
                    int64_t n, int K, int G, float* out, int64_t out_k_stride, int64_t out_g_stride,
                    void* stream);

/*
 * Exact masked percentiles of a UNION of units — several granules, row slabs or processes whose samples form one
 * fit — bit-identical to np.percentile of the concatenated masked samples.  A radix select by 4 passes of 8 bits
 * (most significant first) over the order-preserving u32 keys of the samples; between passes only integer counts
 * cross units and processes, and integer sums do not depend on the order they are added in, so every process ends
 * with the same result.  S series: a unit contributes K planes (x only: S = K) or 2K (x then y: S = 2K).
 *
 *   hsr_union_select_state_bytes   bytes of device state for Q percentiles and S series (0 if out of range);
 *                                  256-byte aligned, reused by every call of one select.
 *   hsr_union_select_hist_doubles  length of the float64 histogram buffer `hist` (8-byte aligned): the per-series /
 *                                  per-target counts of the pass, exact integers below 2^53.
 *   hsr_union_select_begin         starts a select: q [Q] f64 device fractions in [0, 1], Q <= HSR_MAX_PERCENTILES,
 *                                  S <= 65535.  Clears state and hist.
 *   hsr_union_select_count         adds ONE unit to the histograms of pass `pass` (0..3): series k of set 0 is
 *                                  x[k*x_k_stride + i], of set 1 y[k*y_k_stride + i] (y nullable), sample i used iff
 *                                  mask[i] != 0 (mask nullable [n]); n < 2^32 per unit, the union's counts are 64-bit
 *                                  on the device.  Pass 0 counts the top byte of every key per series, and the NaNs;
 *                                  passes 1..3 count the next byte of the keys that carry each target's prefix.
 *                                  On return the stream has `hist` = the sums of every unit counted so far.
 *   hsr_union_select_step          consumes the SUMMED `hist` of the pass: picks the digit of the two ranks
 *                                  (floor / floor + 1 of numpy's virtual index) of every percentile, updates each
 *                                  target's prefix and remaining rank, and clears hist for the next pass.  Pass 0 forms
 *                                  the ranks from the union's sample count n.  *more (host, nullable) = 1 while passes
 *                                  follow; the last pass (3) writes out [S, Q] f64 with numpy's "linear"
 *                                  interpolation (as hsr_masked_percentiles_f64).  A NaN among the union's masked
 *                                  samples, or no sample at all, gives NaN.
 * Sequence, on one stream:
 *     begin(q, Q, S);
 *     for pass = 0, 1, 2, 3:  count(unit, pass) for every local unit (any number, any order);
 *                             SUM all-reduce of hist (hsr_union_select_hist_doubles(Q, S) f64) across processes —
 *                             any f64 SUM all-reduce, e.g. hsr_allreduce_moments; skip it with one process;
 *                             step(pass, &more)
 * Every process makes the same begin / all-reduce / step calls (a process with no unit skips only the counts).
 */
HSR_API size_t hsr_union_select_state_bytes(int Q, int S);
HSR_API int64_t hsr_union_select_hist_doubles(int Q, int S);
HSR_API int hsr_union_select_begin(const double* q, int Q, int S, void* state, double* hist, void* stream);
HSR_API int hsr_union_select_count(const float* x, int64_t x_k_stride, const float* y, int64_t y_k_stride,
                           const uint8_t* mask, int64_t n, int K, int Q, int pass, void* state, double* hist,
                           void* stream);
HSR_API int hsr_union_select_step(int Q, int S, int pass, void* state, double* hist, double* out, int* more,
                          void* stream);

/*
 * hsr_union_select_count_bilinear: hsr_union_select_count for a unit whose K series (x only: S = K) are the VIRTUAL
 * planes bilinear x factor of the coarse planes src (K planes [Hs, Ws] f32, plane stride src_plane_stride): sample i of
 * series k is fine pixel i of hsr_bilinear_upsample_f32(src[k], factor) without nodata (same bits), formed where
 * mask[i] != 0 (mask nullable [Hs*factor, Ws*factor]) and never written.  The fine planes of s2_emit/poly_regression.py
 * :150-161 (2 GB at 10 m for a granule) are not materialised; the 60 m planes stay in L2 across the four passes.
 * factor^2 * Hs * Ws < 2^32 (HSR_ERANGE otherwise).  Takes the place of hsr_union_select_count in the sequence above;
 * begin, step and the all-reduce are unchanged, and units of both kinds may be counted into one select.
 */
HSR_API int hsr_union_select_count_bilinear(const float* src, int64_t src_plane_stride, int64_t Hs, int64_t Ws,
                                    int factor, const uint8_t* mask, int K, int Q, int pass, void* state,
                                    double* hist, void* stream);

/*
 * Optimal-transport targets of fit_ot_poly_rgb, s2_emit/poly_regression.py:31-60.  POT (`import ot`) is an
 * un-vendored, un-pinned dependency of the reference; these entry points follow its published algorithms
 * (ot.dist "sqeuclidean" = |x|^2 + |y|^2 - 2 x.y clamped at 0; ot.sinkhorn = sinkhorn_knopp), all in fp64.
 *
 * hsr_compact_finite_rows: idx = row-major indices of the rows of img [n, C] (f32, interleaved) whose mask byte
 *   is set and whose C channels are all finite — `img[mask]` followed by the finite filter of :33-36;
 *   count[0] = how many.  workspace: hsr_compact_workspace_bytes(n) bytes.
 * hsr_gather_rows_f64: out[r, :] = (f64) img[idx[sel[r]], :] — `X_all[rng.choice(...)]` (:46-47); the index
 *   draw itself (numpy's Generator.choice) is host logic and stays on the host.
 * hsr_sinkhorn_barycentric_f64: X [ns, C], Y [nt, C] f64 -> ybar [ns, C] = (P @ Y) / (P.sum(1) + 1e-32) with
 *   P = sinkhorn_knopp(a = 1/ns, b = 1/nt, M = dist(X, Y), reg, numItermax, stopThr) (:49-56): marginal error
 *   checked every 10th iteration, roll-back to the previous (u, v) on 0 / NaN / Inf.  All iterations are
 *   enqueued at once; convergence is a device-side flag (no host synchronisation).
 *   info: nullable [4] f64 out {iteration whose (u, v) were used, last evaluated marginal error, iteration it
 *   was evaluated at, 1 if stopped by a numerical error}.  workspace: hsr_sinkhorn_workspace_bytes(ns, nt)
 *   bytes, 256-byte aligned (holds the ns x nt fp64 kernel matrix).  C <= 4.
 * hsr_polyfit_moments_f64in: normal-equation moments (layout of hsr_poly_moments_f64) of S series of n fp64
 *   samples stored [n, S] (the columns of X and ybar); solve with hsr_poly_solve_f64 -> np.polyfit of :58-60.
 *
 * The same stage on the K planes of a pair synthesis (PairSynthesizer(targets="ot")), padded or dense:
 * hsr_compact_planes_pair: one count / scan / scatter over the mask and both plane sets x, y (K planes each, plane k
 *   at x + k * x_plane_stride; strides >= n, any value when K = 1).  idx_x = row-major indices of the pixels whose mask
 *   byte is set (mask nullable: every pixel) and whose K x values are all finite, count_x[0] = how many; idx_y /
 *   count_y likewise for y — the two filters of :33-36, independent of each other.  x_stretch / y_stretch: nullable
 *   [K][2] f64 (lo, hi); given, a value is judged after the percentile stretch of color.py:33 (true division, as
 *   hsr_stretch_f32).  n < 2^31, 1 <= K <= HSR_MAX_SRF_BANDS.  workspace: hsr_compact_planes_pair_workspace_bytes(n)
 *   bytes, 256-byte aligned.
 * hsr_gather_planes_f64: out[dst[r], k] = (f64) s(planes[k, idx[sel[r]]]) for r < ns, k < K (out row-major with K
 *   columns; dst nullable: row r), s the stretch of color.py:33 with stretch [K][2] (lo, hi), or none when stretch is
 *   null — the stretched samples carry the bits of hsr_stretch_f32.  Rows of out that no r maps to are not written:
 *   a buffer prefilled with -0.0 (the additive identity of IEEE sums: -0.0 + v == v for every v, +0.0 included) can
 *   hold the rows one rank owns and be SUM-all-reduced into the union's rows bit for bit.
 * hsr_sinkhorn_barycentric_k_f64: hsr_sinkhorn_barycentric_f64 for C <= HSR_MAX_SRF_BANDS channels (same workspace,
 *   same loop).  C <= 4 runs the kernels of hsr_sinkhorn_barycentric_f64, so its results are bit-identical to it.
 */
HSR_API size_t hsr_compact_workspace_bytes(int64_t n);
HSR_API int hsr_compact_finite_rows(const float* img, const uint8_t* mask, int64_t n, int C, void* workspace,
                            int32_t* idx, int64_t* count, void* stream);
HSR_API int hsr_gather_rows_f64(const float* img, const int32_t* idx, const int64_t* sel, int64_t ns, int C,
                        double* out, void* stream);
HSR_API size_t hsr_sinkhorn_workspace_bytes(int ns, int nt);
HSR_API int hsr_sinkhorn_barycentric_f64(const double* X, const double* Y, int ns, int nt, int C, double reg,
                                 int num_iter_max, double stop_thr, void* workspace, double* ybar,
                                 double* info, void* stream);
HSR_API int hsr_polyfit_moments_f64in(const double* x, const double* y, int64_t n, int S, int deg,
                              double* moments, void* stream);
HSR_API size_t hsr_compact_planes_pair_workspace_bytes(int64_t n);
HSR_API int hsr_compact_planes_pair(const float* x, int64_t x_plane_stride, const double* x_stretch, const float* y,
                            int64_t y_plane_stride, const double* y_stretch, const uint8_t* mask, int64_t n,
                            int K, void* workspace, int32_t* idx_x, int64_t* count_x, int32_t* idx_y,
                            int64_t* count_y, void* stream);
HSR_API int hsr_gather_planes_f64(const float* planes, int64_t plane_stride, int K, const int32_t* idx,
                          const int64_t* sel, const int64_t* dst, int64_t ns, const double* stretch, double* out,
                          void* stream);
HSR_API int hsr_sinkhorn_barycentric_k_f64(const double* X, const double* Y, int ns, int nt, int C, double reg,
                                   int num_iter_max, double stop_thr, void* workspace, double* ybar,
                                   double* info, void* stream);

/*
 * Tile validity and uint16 quantisation, tiles_helpers/utils.py (the step after orthorectification in the
 * dataset pipeline), on band-sequential float32 tiles (bands, H, W) as rasterio hands them to the reference.
 *
 * hsr_black_mask_f32 — is_black_mask (:201-220): out[g, i] = 1 iff ALL B bands of pixel i are ~ nodata
 *   (if has_nodata), or ALL ~ masked (-0.01), or ALL |v| < zero_tol.  "~" is np.isclose on a float32 array
 *   against a Python float: |v - f32(y)| <= tol or v == f32(y), with tol = f32(atol + 1e-5 * |y|) computed by
 *   the caller (nodata_tol, masked_tol).  arr: G tiles, band b of tile g at arr + g*g_stride + b*b_stride,
 *   n pixels each.  count: nullable [G] u64, ACCUMULATED number of black pixels per tile (the black fraction
 *   find_valid_paired_tiles thresholds, :282-288).
 * hsr_quantize_u16_f32 — save_tile_pair (:362-373): out = valid ? clip(int32(rint(v * scale)), 0, nodata_u16 - 1)
 *   : nodata_u16, valid = isfinite(v) & (v != nodata) (nodata test only if has_nodata); float32 product, ties
 *   to even.  x, out: n elements (any shape, flattened).
 */
HSR_API int hsr_black_mask_f32(const float* arr, int64_t g_stride, int64_t b_stride, int64_t n, int B, int G,
                       int has_nodata, float nodata, float nodata_tol, float masked, float masked_tol,
                       float zero_tol, uint8_t* out, unsigned long long* count, void* stream);
HSR_API int hsr_quantize_u16_f32(const float* x, int64_t n, int has_nodata, float nodata, float scale,
                         int nodata_u16, uint16_t* out, void* stream);
/*
 * Fused tile export: GLT gather + uint16 quantisation + black mask in ONE pass over the raw cube; the fp32 ortho
 * cube is never written (1.8 GB read + 1.6 GB written instead of 5.0 + 4.8 + 3.2 GB for gather, quantise, mask).
 *   out[b, p] = quantise(ortho[p, b]) as hsr_quantize_u16_f32 does, band-sequential (bands, out_h, out_w) — the layout
 *               of the reference's tiles — plane stride plane_stride elements; invalid GLT pixels quantise `fill`.
 *   black[p]  = is_black_mask of the ortho pixel (all bands ~ nodata | all ~ masked | all |v| < zero_tol), nullable;
 *               tolerances as in hsr_black_mask_f32.
 *   valid, diag, view as in hsr_glt_ortho_f32.  bands >= 32.
 */
HSR_API int hsr_glt_ortho_u16(const float* raw, int64_t raw_h, int64_t raw_w, int bands, int64_t raw_pix_stride,
                      int transpose_raw_yx, const int32_t* glt_x, const int32_t* glt_y,
                      int64_t out_h, int64_t out_w, int64_t glt_row_stride, float fill,
                      float scale, int has_nodata, float nodata, int nodata_u16,
                      uint16_t* out, int64_t plane_stride, uint8_t* valid, uint8_t* black,
                      float nodata_tol, float masked, float masked_tol, float zero_tol,
                      unsigned long long* diag, const hsr_raw_view_t* view, void* stream);
/* out[ty*ntx + tx] = number of set bytes of mask [H, W] inside the non-overlapping tile (ty, tx) of tile_h x tile_w
 * pixels — `emit_black.sum()` per window of find_valid_paired_tiles (tiles_helpers/utils.py:266-288). */
HSR_API int hsr_tile_sums_u8(const uint8_t* mask, int64_t H, int64_t W, int tile_h, int tile_w, int nty, int ntx,
                     uint32_t* out, void* stream);

/*
 * "average" resampling onto a coarser ALIGNED grid with an integer pixel ratio — the notebook's
 * downsample_s2_to_grid (Pairs_EMIT_S2_demo-2.ipynb cell 73; s2_emit/poly_regression.py:110-116) for grids
 * snapped as nc_to_envi snaps them (emit_proj.py:794-797): dst[c, y, x] = mean of the valid pixels of the
 * factor x factor source block (float64 mean -> float32; nodata and NaN excluded; none valid -> 0), then
 * `* scale` in float32 if has_scale.  src: C planes [Hs, Ws] of u8 (src_dtype 0), u16 (1) or f32 (2); the last
 * Hs % factor rows / Ws % factor columns are dropped.  Parity with GDAL itself is unpinned (not installable here).
 */
HSR_API int hsr_block_average_f32(const void* src, int src_dtype, int C, int64_t Hs, int64_t Ws, int64_t src_plane_stride,
                          int factor, int has_nodata, double nodata, int has_scale, float scale,
                          float* dst, int64_t dst_plane_stride, void* stream);

/*
 * Bilinear resampling onto a `factor`-times finer ALIGNED grid — the notebook's reproject_stack_to_grid with
 * Resampling.bilinear (cell 73; s2_emit/poly_regression.py:150-156: pseudo-S2 planes 60 m -> 10 m): 2 x 2 source
 * neighbours of the destination pixel centre, neighbours outside the source / equal to nodata / NaN skipped with the
 * weights renormalised, none usable -> 0.  src: C planes [Hs, Ws] f32; dst: C planes [Hs*factor, Ws*factor] f32.
 * Parity with GDAL itself is unpinned.
 */
HSR_API int hsr_bilinear_upsample_f32(const float* src, int C, int64_t Hs, int64_t Ws, int64_t src_plane_stride, int factor,
                              int has_nodata, float nodata, float* dst, int64_t dst_plane_stride, void* stream);

/*
 * Colour-matched planes at the finer resolution, s2_emit/poly_regression.py:150-162 on K planes, without the fine
 * intermediates.  src: K <= HSR_MAX_SRF_BANDS coarse planes [Hs, Ws] f32 (plane stride src_plane_stride); fine pixel i
 * of plane k is x10[k][i] = hsr_bilinear_upsample_f32(src[k], factor) without nodata (same bits).
 * hsr_bilinear_fine_mask_u8: mask [Hs*factor, Ws*factor] u8 = all_k isfinite(x10[k]) (hsr_fit_mask_u8 with no gate).
 * hsr_bilinear_apply_f32:    dst[k] = xs = x10[k], stretched first with x_stretch (nullable [K][2] f64 (lo, hi), the
 *                            on-the-fly stretch of hsr_poly_solve_apply_f32) on every pixel; where mask10:
 *                            (f32) polyval_f64(coeffs[k], xs) (coeffs [K, deg+1] f64, highest power first); then every
 *                            pixel clipped to [lo, hi] (lo > hi: no clip).  Bit-identical to hsr_bilinear_upsample_f32
 *                            -> hsr_fit_mask_u8 (gate_k < 0) -> hsr_poly_solve_apply_f32 with the moments that gave
 *                            coeffs.  dst: K planes of Hs*factor*Ws*factor, plane stride dst_plane_stride (16-byte
 *                            stores where dst and the stride allow); mask_out nullable: receives mask10.
 */
HSR_API int hsr_bilinear_fine_mask_u8(const float* src, int K, int64_t Hs, int64_t Ws, int64_t src_plane_stride,
                              int factor, uint8_t* mask, void* stream);
HSR_API int hsr_bilinear_apply_f32(const float* src, int K, int64_t Hs, int64_t Ws, int64_t src_plane_stride,
                           int factor, const double* coeffs, int deg, const double* x_stretch, float lo, float hi,
                           float* dst, int64_t dst_plane_stride, uint8_t* mask_out, void* stream);

/*
 * robust_norm / robust_norm_rgb of s2_emit/color.py:6-23, whose results are float64:
 * hsr_stretch_f64: out = clip((f64(x) - lo) / (hi - lo + 1e-12), 0, 1) as float64 (same series layout and [S][2] table as
 * hsr_stretch_f32), NaN wherever mask row g ([G][n], nullable) is 0 — `cc[~mask] = np.nan` (:20).
 * hsr_notnan_mask_u8: out[i] = !isnan(x[i]) (& base[i] if given): the sample set of np.nanpercentile (:7) as the mask
 * of hsr_masked_percentiles_f64.
 */
HSR_API int hsr_stretch_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride, const double* lohi, const uint8_t* mask,
                    int64_t n, int K, int G, double* out, int64_t out_k_stride, int64_t out_g_stride, void* stream);
HSR_API int hsr_notnan_mask_u8(const float* x, const uint8_t* base, int64_t n, uint8_t* out, void* stream);

/*
 * Histogram matching of one channel, s2_emit/color.py:36-61 (_hist_match_channel + the clip of histogram_match_rgb), on
 * SORTED sample arrays (the caller sorts the masked samples; np.unique's value / count tables are implicit in them):
 *   hsr_run_ends_u8     flags[i] = 1 where sorted[i] is the last of a run of equal values (the distinct values of
 *                       np.unique and their cumulative counts i + 1); compacted into ref_run_ends by the caller
 *                       (hsr_compact_finite_rows does it);
 *   hsr_hist_match_f32  masked pixels: q = #(src_sorted <= x) / ns, out = float32(np.interp(q, r_quant, r_values)) with
 *                       r_quant[j] = (ref_run_ends[j] + 1) / nr, r_values[j] = ref_sorted[ref_run_ends[j]], numpy's
 *                       float64 arithmetic; then EVERY pixel is clipped to [0, 1].  Samples are assumed finite.
 */
HSR_API int hsr_run_ends_u8(const float* sorted, int64_t n, uint8_t* flags, void* stream);
HSR_API int hsr_hist_match_f32(const float* src, const uint8_t* mask, int64_t n, const float* src_sorted, int64_t ns,
                       const float* ref_sorted, int64_t nr, const int32_t* ref_run_ends, int64_t nu, float* out,
                       void* stream);

/*
 * Affine colour transfer on OT targets — the tail of ot_match_rgb_sinkhorn_pot (s2_emit/color.py:103-115) after
 * hsr_sinkhorn_barycentric_f64:  W = lstsq([X 1], Ybar)  ((C+1) x C row-major: rows 0..C-1 = A, row C = t), solved
 * from the fp64 normal equations in one CTA (fixed summation order);  out = float32(rgb), and where mask (everywhere if
 * NULL) out = float32(clip(float64(x) @ A + t, lo, hi)) — pixels outside the mask are copied, NOT clipped (:110-115).
 * X, Ybar [ns, C] f64; rgb, out [n, C] f32 interleaved; mask [n]; C <= 4.
 */
HSR_API int hsr_affine_fit_f64(const double* X, const double* Ybar, int64_t ns, int C, double* W, void* stream);
HSR_API int hsr_affine_apply_f32(const float* rgb, const double* W, const uint8_t* mask, int64_t n, int C,
                         float lo, float hi, float* out, void* stream);

/*
 * General grid warp (SURVEY section 8f row 4, general case): what nc_to_envi hands to the subprocess
 *   gdalwarp -t_srs <S2 CRS> -te <snapped extent> -ts cols rows -srcnodata -9999 -dstnodata -9999 -r cubic
 * (EMIT_data/emit_proj.py:876-940): the band-interleaved WGS-84 ortho cube resampled onto the Sentinel-2 UTM grid.
 * Geometry (host doubles, read during the call):
 *   src_gt / dst_gt  GDAL geotransforms (x_ul, x_res, x_rot, y_ul, y_rot, y_res) of the two grids;
 *   utm_zone         0: both grids share one CRS (affine only — the notebook's reproject_stack_to_grid between two
 *                    grids of one UTM zone); 1..60: the destination is WGS-84 / UTM zone utm_zone (EPSG:326zz, or
 *                    327zz with south != 0) and the source is geographic lon / lat in degrees (EPSG:4326);
 *   xscale, yscale   destination size / source-window size per axis (GDAL's dfXScale / dfYScale; <= 0 reads as 1):
 *                    below 1 the filter is widened to ceil(r / scale) taps and its argument scaled (anti-aliasing).
 * Algorithm (restated from GDAL's gdalwarpkernel.cpp and PROJ's tmerc — parity with GDAL / PROJ is UNPINNED, neither
 * is installable in the build image; oracle/warp.py is the checker): destination pixel centre -> source pixel
 * coordinates exactly per pixel (gdalwarp -et 0; inverse transverse Mercator by the Krueger series to n^6, fp64);
 * kernel 2 = cubic convolution (a = -0.5, radius 2), 1 = bilinear (radius 1); taps outside the source or equal to
 * nodata (per band) are skipped and the sum divided by the accumulated weight; a centre outside the source or an
 * accumulated weight < 1e-6 leaves dst_nodata.  NaN is an ordinary value.
 * kernel 0 = nearest neighbour (the source pixel floor(x + 1e-10), floor(y + 1e-10) that holds the destination centre;
 * nodata there leaves dst_nodata) and 3 = "average" (every source pixel touched by the box between the destination
 * pixel's transformed top-left and bottom-right corners, weighted by the fraction covered along each axis, nodata
 * skipped per band, fp64 sums) — what rasterio.warp.reproject is asked for in s2_data/s2_utils.py:546-574 (nearest,
 * bilinear) and by the notebook's downsample_s2_to_grid (average, s2_emit/poly_regression.py:110-116) when the grids
 * are not snapped to an integer ratio; xscale / yscale and the workspace are not used by these two.
 * src [Hs, Ws, bands] f32 with src_pix_stride, dst [Hd, Wd, bands] f32 with dst_pix_stride (elements).  Records
 * padded to a multiple of 4 floats on 16-byte aligned bases take the vector path (pad words of dst are undefined).
 * workspace: hsr_warp_workspace_bytes(Hd, Wd) bytes of 16-byte aligned device memory for the source coordinates of
 * the destination pixels (transformed once by a separate launch); required by kernels 1 and 2 (NULL: HSR_EINVAL).
 */
typedef struct hsr_warp_geo {
    double src_gt[6];
    double dst_gt[6];
    int utm_zone;
    int south;
    double xscale, yscale;
} hsr_warp_geo_t;
HSR_API int hsr_warp_f32(const float* src, int64_t Hs, int64_t Ws, int bands, int64_t src_pix_stride,
                 const hsr_warp_geo_t* geo, int kernel, int has_nodata, float nodata, float dst_nodata,
                 int64_t Hd, int64_t Wd, float* dst, int64_t dst_pix_stride, void* workspace, size_t workspace_bytes,
                 void* stream);
HSR_API size_t hsr_warp_workspace_bytes(int64_t Hd, int64_t Wd);
/* coords[Hd, Wd, 2] = source pixel coordinates (x, y; pixel (i, j) has its centre at (i + 0.5, j + 0.5)) of every
 * destination pixel centre — the transformer of hsr_warp_f32 on its own (tests, diagnostics, footprints). */
HSR_API int hsr_warp_coords_f64(const hsr_warp_geo_t* geo, int64_t Hd, int64_t Wd, double* coords, void* stream);
/*
 * Warp of K planar images onto the Sentinel-2 grid: the pseudo-S2 planes of hsr_glt_srf_f32 instead of the B-band
 * ortho cube.  The SRF contraction and the warp are both linear, and the warp's tap weights are the same for every
 * band wherever a source pixel is all data or all nodata, which the GLT fill is; so warping the K planes gives
 * SRF(warp(cube)).  Tap rule of hsr_warp_f32 (kernel 1 bilinear, 2 cubic; radius ceil(r / scale) per axis below
 * scale 1 with the argument scaled; tap weight = fp32 rounding of the fp64 product wy * wx), except that validity is
 * per source pixel: a tap is skipped when its weight is 0 (even over a NaN), when it is outside the source or when
 * src_valid is 0.  The K sums and the weight sum are accumulated in fp64 and dst[k] = f32(acc[k] / ws).  A centre
 * outside the source or ws < 1e-6: dst[k] = fill_out[k] and dst_valid = 0.  Non-finite values propagate as in the
 * per-band warp.  fit_mask = dst_valid & all_k isfinite(dst[k]) & (dst[gate_k] > gate_gt) (gate_k < 0: no gate),
 * the rule hsr_glt_srf_f32 writes.
 *   src       [K] planes of Hs * Ws f32, plane k at src + k * src_plane_stride (>= Hs * Ws unless K == 1);
 *   src_valid [Hs, Ws] u8, 1 = the pixel's taps may be used (the GLT valid mask);
 *   coords    [Hd, Wd, 2] f64 from hsr_warp_coords_f64 (16-byte aligned); required;
 *   geo       only xscale / yscale are read (<= 0 reads as 1);
 *   fill_out  [K] f32 device; dst [K] planes of Hd * Wd with dst_plane_stride; dst_valid, fit_mask [Hd, Wd] u8,
 *             both nullable.
 * Exactness: equal to pseudo_s2_srf_integral(warp(glt_ortho(raw))) in exact arithmetic; in fp, planes within
 * 1e-5 * C_k + 1e-7 where C_k = sum_t |w_t| |v_tk| / |sum_t w_t| (the conditioning of the renormalised sum), identical
 * coverage and NaN / Inf patterns, fill_out where uncovered.  Deviation: a GLT-valid raw spectrum holding the nodata
 * value in some or all of its bands is used as data (the per-band warp skips it for those bands).
 * HSR_EINVAL: K outside 1..16, NULL coords (or src / dst / src_valid / fill_out / geo), kernel not 1 / 2, a filter
 * radius beyond 8 taps (scale < 0.25 cubic, < 0.125 bilinear), plane strides below the plane size, gate_k >= K.
 */
HSR_API int hsr_warp_planes_f32(const float* src, int64_t Hs, int64_t Ws, int K, int64_t src_plane_stride,
                                const uint8_t* src_valid, const double* coords, const hsr_warp_geo_t* geo, int kernel,
                                const float* fill_out, int gate_k, float gate_gt, int64_t Hd, int64_t Wd, float* dst,
                                int64_t dst_plane_stride, uint8_t* dst_valid, uint8_t* fit_mask, void* stream);

/*
 * Row slabs of the Sentinel-2 grid (a mosaic target dealt to ranks by rows).  Call order for one band of target rows
 * [row0, row0 + rows): hsr_warp_coords_rows_f64 -> hsr_warp_src_row_range (source = ortho rows [o0, o1)) ->
 * hsr_glt_row_range on GLT rows [o0, o1) (raw rows to stage) -> hsr_glt_srf_f32 with an hsr_raw_view_t ->
 * hsr_warp_planes_window_f32 with src_row0 = o0, src_rows = o1 - o0.
 *
 * hsr_warp_coords_rows_f64: coords[r - row0] for destination rows r in [row0, row0 + rows), coords [rows, Wd, 2] f64.
 * The transform takes the absolute row (r + 0.5), so the band is bit-identical to those rows of hsr_warp_coords_f64.
 */
HSR_API int hsr_warp_coords_rows_f64(const hsr_warp_geo_t* geo, int64_t row0, int64_t rows, int64_t Wd, double* coords,
                                     void* stream);
/*
 * hsr_warp_src_row_range: the source rows that hsr_warp_planes_f32 reads for the destination pixels of coords
 * [rows, Wd, 2] (16-byte aligned).  Over every pixel whose centre is inside the Hs x Ws source: range[0] =
 * min(floor(py - 0.5) + 1 - ry), range[1] = max(floor(py - 0.5) + 1 + ry), both clipped to [0, Hs), with ry the
 * plane warp's row radius for `kernel` (1 / 2) and geo->yscale (only xscale / yscale are read).  Conservative: taps
 * of zero weight and invalid source pixels are included.  ACCUMULATED with min / max like hsr_glt_row_range: the
 * caller initialises range to {UINT64_MAX, 0}; an untouched range means no centre is inside the source.
 */
HSR_API int hsr_warp_src_row_range(const double* coords, int64_t rows, int64_t Wd, int64_t Hs, int64_t Ws,
                                   const hsr_warp_geo_t* geo, int kernel, unsigned long long* range /*[2] u64*/,
                                   void* stream);
/*
 * hsr_warp_planes_window_f32: hsr_warp_planes_f32 over a window of source rows.  src / src_valid hold only rows
 * [src_row0, src_row0 + src_rows) of the logical Hs x Ws source (plane stride >= src_rows * Ws unless K == 1); Hs
 * stays the logical height, so the "centre outside the source" test, the tap bounds, the weights and the fp64 sums are
 * those of the unwindowed call, and where the window holds every row a pixel's non-zero-weight taps reach, its output
 * is bit-identical to hsr_warp_planes_f32 on the whole source.  A non-zero-weight tap in a row outside the window is
 * skipped and its destination pixel counted in *outside (nullable, u64, ACCUMULATED): the caller must treat a non-zero
 * count as an error (it sized the window wrongly), as it does diag[3] of a raw view.  src_rows = 0 is allowed (src /
 * src_valid may then be NULL): nothing is read and every pixel gets fill_out, dst_valid = 0 and fit_mask = 0.
 * hsr_warp_planes_f32 is this call with src_row0 = 0, src_rows = Hs and no counter.
 * HSR_EINVAL: as hsr_warp_planes_f32, and a window outside [0, Hs).
 */
HSR_API int hsr_warp_planes_window_f32(const float* src, int64_t Hs, int64_t Ws, int K, int64_t src_plane_stride,
                                       const uint8_t* src_valid, int64_t src_row0, int64_t src_rows,
                                       const double* coords, const hsr_warp_geo_t* geo, int kernel,
                                       const float* fill_out, int gate_k, float gate_gt, int64_t Hd, int64_t Wd,
                                       float* dst, int64_t dst_plane_stride, uint8_t* dst_valid, uint8_t* fit_mask,
                                       unsigned long long* outside, void* stream);

/*
 * Peer blocks for hsr_exchange_t.  hsr_peer_alloc creates (cudaMalloc + zero) this rank's block — the one
 * persistent allocation the library makes, the analogue of a communicator; hsr_ipc_export / hsr_ipc_import wrap
 * cudaIpcGetMemHandle / cudaIpcOpenMemHandle (lazy peer access) so that the processes of one node can map each
 * other's blocks; the 64-byte handles travel through whatever the host uses (torch.distributed here).
 */
HSR_API size_t hsr_peer_block_bytes(void);
HSR_API int hsr_peer_alloc(void** dptr);
HSR_API int hsr_peer_free(void* dptr);
HSR_API int hsr_ipc_export(const void* dptr, unsigned char* handle /*[HSR_IPC_HANDLE_BYTES]*/);
HSR_API int hsr_ipc_import(const unsigned char* handle, void** dptr);
HSR_API int hsr_ipc_close(void* dptr);
/* Synchronises `stream`, copies the block's sticky status word to *status (host memory) and returns HSR_EPEER
 * when HSR_PEER_TIMEOUT is set (hsr_last_error says why), HSR_OK otherwise. */
HSR_API int hsr_peer_status(const void* my_block, unsigned int* status, void* stream);

/*
 * The generic form of the one collective of the path (SURVEY 8b / 8e): in-place SUM all-reduce of `count` float64
 * moments over an NCCL communicator the HOST created (ncclComm_t passed as void*), i.e.
 * ncclAllReduce(moments, moments, count, ncclDouble, ncclSum, comm, stream).  For hosts that do not go through
 * torch.distributed and do not want the peer-memory exchange (several nodes, no CUDA IPC).  libnccl.so.2 is
 * resolved at the first call — the copy already loaded into the process if there is one — so the library itself
 * has no link-time dependency on NCCL; HSR_ENCCL when it cannot be loaded or the call fails.
 * Sits between hsr_fit_moments_f64 (exchange = NULL) and hsr_poly_solve_apply_f32 (exchange = NULL).
 */
HSR_API int hsr_allreduce_moments(double* moments, int64_t count, void* nccl_comm, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HSR_B200_H */
