// abi.cu — the extern "C" surface of libhsr_b200.so (declared in include/hsr_b200.h) and the
// thread-local error string.  Everything here is argument plumbing; kernels live in
// glt_stream.cu and poly.cu.
#include <stdarg.h>
#include <string.h>

#include "hsr_common.cuh"

namespace hsr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return (int)e;
}

int current_device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return 0;
    return dev < HSR_MAX_DEVICES ? dev : HSR_MAX_DEVICES - 1;
}

static int cached_attr(cudaDeviceAttr attr, int* cache, int dflt) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return dflt;
    const bool slot = dev >= 0 && dev < HSR_MAX_DEVICES;
    if (slot) {
        const int c = __atomic_load_n(&cache[dev], __ATOMIC_RELAXED);
        if (c > 0) return c;
    }
    int n = 0;
    if (cudaDeviceGetAttribute(&n, attr, dev) != cudaSuccess || n <= 0) return dflt;
    if (slot) __atomic_store_n(&cache[dev], n, __ATOMIC_RELAXED);
    return n;
}

int device_sm_count() {
    static int cache[HSR_MAX_DEVICES];
    return cached_attr(cudaDevAttrMultiProcessorCount, cache, 148);
}

int device_max_smem_optin() {
    static int cache[HSR_MAX_DEVICES];
    return cached_attr(cudaDevAttrMaxSharedMemoryPerBlockOptin, cache, 0);
}

int glt_ortho_impl(const float*, long long, long long, int, long long, int, const int32_t*, const int32_t*, long long,
                   long long, long long, float, float*, long long, uint8_t*, unsigned long long*, const hsr_raw_view_t*,
                   cudaStream_t);
int glt_srf_impl(const float*, long long, long long, int, long long, int, const int32_t*, const int32_t*, long long,
                 long long, long long, float, const float*, const float*, int, float*, long long, float*, long long,
                 uint8_t*, unsigned long long*, uint8_t*, int, float, const hsr_raw_view_t*, cudaStream_t);
int glt_row_range_impl(const int32_t*, const int32_t*, long long, long long, long long, long long, long long, int,
                       unsigned long long*, cudaStream_t);
int srf_impl(const float*, long long, int, long long, const float*, int, float*, long long, uint8_t*, int, float,
             cudaStream_t);
int glt_ortho_u16_impl(const float*, long long, long long, int, long long, int, const int32_t*, const int32_t*, long long,
                       long long, long long, float, float, int, float, int, uint16_t*, long long, uint8_t*, uint8_t*,
                       float, float, float, float, unsigned long long*, const hsr_raw_view_t*, cudaStream_t);
int poly_moments_impl(const float*, long long, long long, const float*, long long, long long, const uint8_t*,
                      long long, long long, long long, int, int, double*, double*, cudaStream_t);
int poly_solve_impl(const double*, int, int, long long, double*, cudaStream_t);
int poly_apply_impl(const float*, long long, long long, const double*, const uint8_t*, long long, long long, long long,
                    int, int, float, float, float*, long long, long long, cudaStream_t);
int fit_mask_impl(const float*, long long, long long, const float*, long long, long long, long long, int, int,
                  const uint8_t*, int, float, uint8_t*, cudaStream_t);
size_t poly_moments_workspace(long long n, int K, int deg);
int fit_moments_impl(const float*, long long, long long, const float*, long long, long long, const uint8_t*, long long,
                     int, int, int, int, float, int, const double*, const double*, uint8_t*, double*, double*,
                     const hsr_exchange_t*, cudaStream_t);
int block_average_impl(const void*, int, int, long long, long long, long long, int, int, double, int, float, float*,
                       long long, cudaStream_t);
int bilinear_upsample_impl(const float*, int, long long, long long, long long, int, int, float, float*, long long,
                           cudaStream_t);
int bilinear_fine_mask_impl(const float*, int, long long, long long, long long, int, uint8_t*, cudaStream_t);
int bilinear_apply_impl(const float*, int, long long, long long, long long, int, const double*, int, const double*, float,
                        float, float*, long long, uint8_t*, cudaStream_t);
int warp_impl(const float*, long long, long long, int, long long, const hsr_warp_geo_t*, int, int, float, float,
              long long, long long, float*, long long, void*, size_t, cudaStream_t);
size_t warp_workspace(long long, long long);
int warp_coords_impl(const hsr_warp_geo_t*, long long, long long, double*, cudaStream_t);
int warp_coords_rows_impl(const hsr_warp_geo_t*, long long, long long, long long, double*, cudaStream_t);
int warp_src_row_range_impl(const double*, long long, long long, long long, long long, const hsr_warp_geo_t*, int,
                            unsigned long long*, cudaStream_t);
int warp_planes_impl(const float*, long long, long long, int, long long, const uint8_t*, const double*,
                     const hsr_warp_geo_t*, int, const float*, int, float, long long, long long, float*, long long,
                     uint8_t*, uint8_t*, cudaStream_t);
int warp_planes_window_impl(const float*, long long, long long, int, long long, const uint8_t*, long long, long long,
                            const double*, const hsr_warp_geo_t*, int, const float*, int, float, long long, long long,
                            float*, long long, uint8_t*, uint8_t*, unsigned long long*, cudaStream_t);
int affine_fit_impl(const double*, const double*, long long, int, double*, cudaStream_t);
int affine_apply_impl(const float*, const double*, const uint8_t*, long long, int, float, float, float*, cudaStream_t);
int stretch64_impl(const float*, long long, long long, const double*, const uint8_t*, long long, int, int, double*,
                   long long, long long, cudaStream_t);
int notnan_mask_impl(const float*, const uint8_t*, long long, uint8_t*, cudaStream_t);
int run_ends_impl(const float*, long long, uint8_t*, cudaStream_t);
int hist_match_impl(const float*, const uint8_t*, long long, const float*, long long, const float*, long long, const int*,
                    long long, float*, cudaStream_t);
size_t peer_block_bytes();
int peer_alloc_impl(void**);
int peer_free_impl(void*);
int ipc_export_impl(const void*, unsigned char*);
int ipc_import_impl(const unsigned char*, void**);
int ipc_close_impl(void*);
int peer_status_impl(const void*, unsigned int*, cudaStream_t);
int moments_sum_impl(const double*, int, long long, double*, const hsr_exchange_t*, cudaStream_t);
int allreduce_moments_impl(double*, long long, void*, cudaStream_t);
size_t fit_moments_workspace(long long n, int K, int G, int deg);
int poly_solve_apply_impl(const float*, long long, long long, const double*, const uint8_t*, long long, int, int, int,
                          long long, float, float, const double*, double*, float*, long long, long long,
                          const hsr_exchange_t*, double*, cudaStream_t);

size_t percentiles_workspace(long long n, int K, int G, int nsets);
int masked_percentiles_impl(const float*, long long, long long, const float*, long long, long long, const uint8_t*,
                            long long, int, int, const double*, int, void*, double*, double*, cudaStream_t);
int stretch_impl(const float*, long long, long long, const double*, long long, int, int, float*, long long, long long,
                 cudaStream_t);
size_t union_state_bytes(int Q, int S);
long long union_hist_doubles(int Q, int S);
int union_begin_impl(const double*, int, int, void*, double*, cudaStream_t);
int union_count_impl(const float*, long long, const float*, long long, const uint8_t*, long long, int, int, int, void*,
                     double*, cudaStream_t);
int union_count_bilinear_impl(const float*, long long, long long, long long, int, const uint8_t*, int, int, int, void*,
                              double*, cudaStream_t);
int union_step_impl(int, int, int, void*, double*, double*, int*, cudaStream_t);

size_t compact_workspace(long long n);
int compact_finite_rows_impl(const float*, const uint8_t*, long long, int, void*, int*, long long*, cudaStream_t);
int gather_rows_impl(const float*, const int*, const long long*, long long, int, double*, cudaStream_t);
size_t sinkhorn_workspace(int ns, int nt);
int sinkhorn_barycentric_impl(const double*, const double*, int, int, int, double, int, double, void*, double*, double*,
                              cudaStream_t);
size_t compact_planes_pair_workspace(long long n);
int compact_planes_pair_impl(const float*, long long, const double*, const float*, long long, const double*,
                             const uint8_t*, long long, int, void*, int*, long long*, int*, long long*, cudaStream_t);
int gather_planes_impl(const float*, long long, int, const int*, const long long*, const long long*, long long,
                       const double*, double*, cudaStream_t);
int sinkhorn_barycentric_k_impl(const double*, const double*, int, int, int, double, int, double, void*, double*,
                                double*, cudaStream_t);
int polyfit_f64_moments_impl(const double*, const double*, long long, int, int, double*, cudaStream_t);

int black_mask_impl(const float*, long long, long long, long long, int, int, int, float, float, float, float, float,
                    uint8_t*, unsigned long long*, cudaStream_t);
int quantize_u16_impl(const float*, long long, int, float, float, int, uint16_t*, cudaStream_t);
int tile_sums_impl(const uint8_t*, long long, long long, int, int, int, int, unsigned int*, cudaStream_t);

}  // namespace hsr

extern "C" {

int hsr_version(void) { return HSR_ABI_VERSION; }

const char* hsr_last_error(void) { return hsr::g_err; }

int hsr_glt_ortho_f32(const float* raw, int64_t raw_h, int64_t raw_w, int bands, int64_t raw_pix_stride,
                      int transpose_raw_yx, const int32_t* glt_x, const int32_t* glt_y, int64_t out_h, int64_t out_w,
                      int64_t glt_row_stride, float fill, float* out, int64_t out_pix_stride, uint8_t* valid,
                      unsigned long long* diag, const hsr_raw_view_t* view, void* stream) {
    return hsr::glt_ortho_impl(raw, raw_h, raw_w, bands, raw_pix_stride, transpose_raw_yx, glt_x, glt_y, out_h, out_w,
                               glt_row_stride, fill, out, out_pix_stride, valid, diag, view, (cudaStream_t)stream);
}

int hsr_glt_srf_f32(const float* raw, int64_t raw_h, int64_t raw_w, int bands, int64_t raw_pix_stride,
                    int transpose_raw_yx, const int32_t* glt_x, const int32_t* glt_y, int64_t out_h, int64_t out_w,
                    int64_t glt_row_stride, float fill, const float* W, const float* fill_out, int K,
                    float* bands_out, int64_t bands_plane_stride, float* ortho_out, int64_t out_pix_stride,
                    uint8_t* valid, unsigned long long* diag, uint8_t* fit_mask, int gate_k, float gate_gt,
                    const hsr_raw_view_t* view, void* stream) {
    return hsr::glt_srf_impl(raw, raw_h, raw_w, bands, raw_pix_stride, transpose_raw_yx, glt_x, glt_y, out_h, out_w,
                             glt_row_stride, fill, W, fill_out, K, bands_out, bands_plane_stride, ortho_out,
                             out_pix_stride, valid, diag, fit_mask, gate_k, gate_gt, view, (cudaStream_t)stream);
}

int hsr_glt_ortho_u16(const float* raw, int64_t raw_h, int64_t raw_w, int bands, int64_t raw_pix_stride,
                      int transpose_raw_yx, const int32_t* glt_x, const int32_t* glt_y, int64_t out_h, int64_t out_w,
                      int64_t glt_row_stride, float fill, float scale, int has_nodata, float nodata, int nodata_u16,
                      uint16_t* out, int64_t plane_stride, uint8_t* valid, uint8_t* black, float nodata_tol, float masked,
                      float masked_tol, float zero_tol, unsigned long long* diag, const hsr_raw_view_t* view,
                      void* stream) {
    return hsr::glt_ortho_u16_impl(raw, raw_h, raw_w, bands, raw_pix_stride, transpose_raw_yx, glt_x, glt_y, out_h, out_w,
                                   glt_row_stride, fill, scale, has_nodata, nodata, nodata_u16, out, plane_stride, valid,
                                   black, nodata_tol, masked, masked_tol, zero_tol, diag, view, (cudaStream_t)stream);
}

int hsr_glt_row_range(const int32_t* glt_x, const int32_t* glt_y, int64_t out_h, int64_t out_w, int64_t glt_row_stride,
                      int64_t raw_h, int64_t raw_w, int transpose_raw_yx, unsigned long long* range, void* stream) {
    return hsr::glt_row_range_impl(glt_x, glt_y, out_h, out_w, glt_row_stride, raw_h, raw_w, transpose_raw_yx, range,
                                   (cudaStream_t)stream);
}

int hsr_srf_f32(const float* cube, int64_t n_pix, int bands, int64_t pix_stride, const float* W, int K,
                float* bands_out, int64_t bands_plane_stride, uint8_t* fit_mask, int gate_k, float gate_gt,
                void* stream) {
    return hsr::srf_impl(cube, n_pix, bands, pix_stride, W, K, bands_out, bands_plane_stride, fit_mask, gate_k,
                         gate_gt, (cudaStream_t)stream);
}

int hsr_poly_moments_f64(const float* x, int64_t x_k_stride, int64_t x_n_stride, const float* y, int64_t y_k_stride,
                         int64_t y_n_stride, const uint8_t* mask, int64_t mask_k_div, int64_t mask_k_mod, int64_t n,
                         int K, int deg, double* partial, double* moments, void* stream) {
    return hsr::poly_moments_impl(x, x_k_stride, x_n_stride, y, y_k_stride, y_n_stride, mask, mask_k_div, mask_k_mod,
                                  n, K, deg, partial, moments, (cudaStream_t)stream);
}

int hsr_poly_solve_f64(const double* moments, int K, int deg, int64_t min_count, double* coeffs, void* stream) {
    return hsr::poly_solve_impl(moments, K, deg, min_count, coeffs, (cudaStream_t)stream);
}

int hsr_poly_apply_f32(const float* x, int64_t x_k_stride, int64_t x_n_stride, const double* coeffs,
                       const uint8_t* mask, int64_t mask_k_div, int64_t mask_k_mod, int64_t n, int K, int deg,
                       float lo, float hi, float* out, int64_t out_k_stride, int64_t out_n_stride, void* stream) {
    return hsr::poly_apply_impl(x, x_k_stride, x_n_stride, coeffs, mask, mask_k_div, mask_k_mod, n, K, deg, lo, hi,
                                out, out_k_stride, out_n_stride, (cudaStream_t)stream);
}

int hsr_fit_mask_u8(const float* x, int64_t x_k_stride, int64_t x_g_stride, const float* y, int64_t y_k_stride,
                    int64_t y_g_stride, int64_t n, int K, int G, const uint8_t* valid, int gate_k, float gate_gt,
                    uint8_t* mask, void* stream) {
    return hsr::fit_mask_impl(x, x_k_stride, x_g_stride, y, y_k_stride, y_g_stride, n, K, G, valid, gate_k, gate_gt,
                              mask, (cudaStream_t)stream);
}

int hsr_fit_moments_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride, const float* y, int64_t y_k_stride,
                        int64_t y_g_stride, const uint8_t* valid, int64_t n, int K, int G, int deg, int gate_k,
                        float gate_gt, int flags, const double* x_stretch, const double* y_stretch, uint8_t* mask,
                        double* partial, double* moments, const hsr_exchange_t* exchange, void* stream) {
    return hsr::fit_moments_impl(x, x_k_stride, x_g_stride, y, y_k_stride, y_g_stride, valid, n, K, G, deg, gate_k,
                                 gate_gt, flags, x_stretch, y_stretch, mask, partial, moments, exchange,
                                 (cudaStream_t)stream);
}

size_t hsr_fit_moments_workspace_bytes(int64_t n, int K, int G, int deg) {
    return hsr::fit_moments_workspace(n, K, G, deg);
}

int hsr_poly_solve_apply_f32(const float* x, int64_t x_k_stride, int64_t x_g_stride, const double* moments,
                             const uint8_t* mask, int64_t n, int K, int G, int deg, int64_t min_count, float lo,
                             float hi, const double* x_stretch, double* coeffs, float* out, int64_t out_k_stride,
                             int64_t out_g_stride, const hsr_exchange_t* exchange, double* moments_out, void* stream) {
    return hsr::poly_solve_apply_impl(x, x_k_stride, x_g_stride, moments, mask, n, K, G, deg, min_count, lo, hi,
                                      x_stretch, coeffs, out, out_k_stride, out_g_stride, exchange, moments_out,
                                      (cudaStream_t)stream);
}

int hsr_moments_sum_f64(const double* per_unit, int units, int64_t count, double* out, const hsr_exchange_t* exchange,
                        void* stream) {
    return hsr::moments_sum_impl(per_unit, units, count, out, exchange, (cudaStream_t)stream);
}

size_t hsr_percentiles_workspace_bytes(int64_t n, int K, int G, int nsets) {
    return hsr::percentiles_workspace(n, K, G, nsets);
}

int hsr_masked_percentiles_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride, const uint8_t* mask, int64_t n,
                               int K, int G, const double* q, int Q, void* workspace, double* out, void* stream) {
    return hsr::masked_percentiles_impl(x, x_k_stride, x_g_stride, nullptr, 0, 0, mask, n, K, G, q, Q, workspace, out,
                                        nullptr, (cudaStream_t)stream);
}

int hsr_masked_percentiles_pair_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride, const float* y,
                                    int64_t y_k_stride, int64_t y_g_stride, const uint8_t* mask, int64_t n, int K, int G,
                                    const double* q, int Q, void* workspace, double* out_x, double* out_y, void* stream) {
    return hsr::masked_percentiles_impl(x, x_k_stride, x_g_stride, y, y_k_stride, y_g_stride, mask, n, K, G, q, Q, workspace,
                                        out_x, out_y, (cudaStream_t)stream);
}

int hsr_stretch_f32(const float* x, int64_t x_k_stride, int64_t x_g_stride, const double* lohi, int64_t n, int K,
                    int G, float* out, int64_t out_k_stride, int64_t out_g_stride, void* stream) {
    return hsr::stretch_impl(x, x_k_stride, x_g_stride, lohi, n, K, G, out, out_k_stride, out_g_stride,
                             (cudaStream_t)stream);
}

size_t hsr_union_select_state_bytes(int Q, int S) { return hsr::union_state_bytes(Q, S); }

int64_t hsr_union_select_hist_doubles(int Q, int S) { return hsr::union_hist_doubles(Q, S); }

int hsr_union_select_begin(const double* q, int Q, int S, void* state, double* hist, void* stream) {
    return hsr::union_begin_impl(q, Q, S, state, hist, (cudaStream_t)stream);
}

int hsr_union_select_count(const float* x, int64_t x_k_stride, const float* y, int64_t y_k_stride, const uint8_t* mask,
                           int64_t n, int K, int Q, int pass, void* state, double* hist, void* stream) {
    return hsr::union_count_impl(x, x_k_stride, y, y_k_stride, mask, n, K, Q, pass, state, hist, (cudaStream_t)stream);
}

int hsr_union_select_count_bilinear(const float* src, int64_t src_plane_stride, int64_t Hs, int64_t Ws, int factor,
                                    const uint8_t* mask, int K, int Q, int pass, void* state, double* hist,
                                    void* stream) {
    return hsr::union_count_bilinear_impl(src, src_plane_stride, Hs, Ws, factor, mask, K, Q, pass, state, hist,
                                          (cudaStream_t)stream);
}

int hsr_union_select_step(int Q, int S, int pass, void* state, double* hist, double* out, int* more, void* stream) {
    return hsr::union_step_impl(Q, S, pass, state, hist, out, more, (cudaStream_t)stream);
}

size_t hsr_compact_workspace_bytes(int64_t n) { return hsr::compact_workspace(n); }

int hsr_compact_finite_rows(const float* img, const uint8_t* mask, int64_t n, int C, void* workspace, int32_t* idx,
                            int64_t* count, void* stream) {
    return hsr::compact_finite_rows_impl(img, mask, n, C, workspace, idx, reinterpret_cast<long long*>(count),
                                         (cudaStream_t)stream);
}

int hsr_gather_rows_f64(const float* img, const int32_t* idx, const int64_t* sel, int64_t ns, int C, double* out,
                        void* stream) {
    return hsr::gather_rows_impl(img, idx, reinterpret_cast<const long long*>(sel), ns, C, out, (cudaStream_t)stream);
}

size_t hsr_sinkhorn_workspace_bytes(int ns, int nt) { return hsr::sinkhorn_workspace(ns, nt); }

int hsr_sinkhorn_barycentric_f64(const double* X, const double* Y, int ns, int nt, int C, double reg, int num_iter_max,
                                 double stop_thr, void* workspace, double* ybar, double* info, void* stream) {
    return hsr::sinkhorn_barycentric_impl(X, Y, ns, nt, C, reg, num_iter_max, stop_thr, workspace, ybar, info,
                                          (cudaStream_t)stream);
}

size_t hsr_compact_planes_pair_workspace_bytes(int64_t n) { return hsr::compact_planes_pair_workspace(n); }

int hsr_compact_planes_pair(const float* x, int64_t x_plane_stride, const double* x_stretch, const float* y,
                            int64_t y_plane_stride, const double* y_stretch, const uint8_t* mask, int64_t n, int K,
                            void* workspace, int32_t* idx_x, int64_t* count_x, int32_t* idx_y, int64_t* count_y,
                            void* stream) {
    return hsr::compact_planes_pair_impl(x, x_plane_stride, x_stretch, y, y_plane_stride, y_stretch, mask, n, K, workspace,
                                         idx_x, reinterpret_cast<long long*>(count_x), idx_y,
                                         reinterpret_cast<long long*>(count_y), (cudaStream_t)stream);
}

int hsr_gather_planes_f64(const float* planes, int64_t plane_stride, int K, const int32_t* idx, const int64_t* sel,
                          const int64_t* dst, int64_t ns, const double* stretch, double* out, void* stream) {
    return hsr::gather_planes_impl(planes, plane_stride, K, idx, reinterpret_cast<const long long*>(sel),
                                   reinterpret_cast<const long long*>(dst), ns, stretch, out, (cudaStream_t)stream);
}

int hsr_sinkhorn_barycentric_k_f64(const double* X, const double* Y, int ns, int nt, int C, double reg,
                                   int num_iter_max, double stop_thr, void* workspace, double* ybar, double* info,
                                   void* stream) {
    return hsr::sinkhorn_barycentric_k_impl(X, Y, ns, nt, C, reg, num_iter_max, stop_thr, workspace, ybar, info,
                                            (cudaStream_t)stream);
}

int hsr_polyfit_moments_f64in(const double* x, const double* y, int64_t n, int S, int deg, double* moments,
                              void* stream) {
    return hsr::polyfit_f64_moments_impl(x, y, n, S, deg, moments, (cudaStream_t)stream);
}

int hsr_black_mask_f32(const float* arr, int64_t g_stride, int64_t b_stride, int64_t n, int B, int G, int has_nodata,
                       float nodata, float nodata_tol, float masked, float masked_tol, float zero_tol, uint8_t* out,
                       unsigned long long* count, void* stream) {
    return hsr::black_mask_impl(arr, g_stride, b_stride, n, B, G, has_nodata, nodata, nodata_tol, masked, masked_tol,
                                zero_tol, out, count, (cudaStream_t)stream);
}

int hsr_quantize_u16_f32(const float* x, int64_t n, int has_nodata, float nodata, float scale, int nodata_u16,
                         uint16_t* out, void* stream) {
    return hsr::quantize_u16_impl(x, n, has_nodata, nodata, scale, nodata_u16, out, (cudaStream_t)stream);
}

int hsr_tile_sums_u8(const uint8_t* mask, int64_t H, int64_t W, int tile_h, int tile_w, int nty, int ntx, uint32_t* out,
                     void* stream) {
    return hsr::tile_sums_impl(mask, H, W, tile_h, tile_w, nty, ntx, out, (cudaStream_t)stream);
}

int hsr_block_average_f32(const void* src, int src_dtype, int C, int64_t Hs, int64_t Ws, int64_t src_plane_stride, int factor,
                          int has_nodata, double nodata, int has_scale, float scale, float* dst, int64_t dst_plane_stride,
                          void* stream) {
    return hsr::block_average_impl(src, src_dtype, C, Hs, Ws, src_plane_stride, factor, has_nodata, nodata, has_scale, scale,
                                   dst, dst_plane_stride, (cudaStream_t)stream);
}

int hsr_bilinear_upsample_f32(const float* src, int C, int64_t Hs, int64_t Ws, int64_t src_plane_stride, int factor,
                              int has_nodata, float nodata, float* dst, int64_t dst_plane_stride, void* stream) {
    return hsr::bilinear_upsample_impl(src, C, Hs, Ws, src_plane_stride, factor, has_nodata, nodata, dst, dst_plane_stride,
                                       (cudaStream_t)stream);
}

int hsr_bilinear_fine_mask_u8(const float* src, int K, int64_t Hs, int64_t Ws, int64_t src_plane_stride, int factor,
                              uint8_t* mask, void* stream) {
    return hsr::bilinear_fine_mask_impl(src, K, Hs, Ws, src_plane_stride, factor, mask, (cudaStream_t)stream);
}

int hsr_bilinear_apply_f32(const float* src, int K, int64_t Hs, int64_t Ws, int64_t src_plane_stride, int factor,
                           const double* coeffs, int deg, const double* x_stretch, float lo, float hi, float* dst,
                           int64_t dst_plane_stride, uint8_t* mask_out, void* stream) {
    return hsr::bilinear_apply_impl(src, K, Hs, Ws, src_plane_stride, factor, coeffs, deg, x_stretch, lo, hi, dst,
                                    dst_plane_stride, mask_out, (cudaStream_t)stream);
}

int hsr_warp_f32(const float* src, int64_t Hs, int64_t Ws, int bands, int64_t src_pix_stride, const hsr_warp_geo_t* geo,
                 int kernel, int has_nodata, float nodata, float dst_nodata, int64_t Hd, int64_t Wd, float* dst,
                 int64_t dst_pix_stride, void* workspace, size_t workspace_bytes, void* stream) {
    return hsr::warp_impl(src, Hs, Ws, bands, src_pix_stride, geo, kernel, has_nodata, nodata, dst_nodata, Hd, Wd, dst,
                          dst_pix_stride, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t hsr_warp_workspace_bytes(int64_t Hd, int64_t Wd) { return hsr::warp_workspace(Hd, Wd); }

int hsr_warp_coords_f64(const hsr_warp_geo_t* geo, int64_t Hd, int64_t Wd, double* coords, void* stream) {
    return hsr::warp_coords_impl(geo, Hd, Wd, coords, (cudaStream_t)stream);
}

int hsr_warp_planes_f32(const float* src, int64_t Hs, int64_t Ws, int K, int64_t src_plane_stride,
                        const uint8_t* src_valid, const double* coords, const hsr_warp_geo_t* geo, int kernel,
                        const float* fill_out, int gate_k, float gate_gt, int64_t Hd, int64_t Wd, float* dst,
                        int64_t dst_plane_stride, uint8_t* dst_valid, uint8_t* fit_mask, void* stream) {
    return hsr::warp_planes_impl(src, Hs, Ws, K, src_plane_stride, src_valid, coords, geo, kernel, fill_out, gate_k,
                                 gate_gt, Hd, Wd, dst, dst_plane_stride, dst_valid, fit_mask, (cudaStream_t)stream);
}

int hsr_warp_coords_rows_f64(const hsr_warp_geo_t* geo, int64_t row0, int64_t rows, int64_t Wd, double* coords,
                             void* stream) {
    return hsr::warp_coords_rows_impl(geo, row0, rows, Wd, coords, (cudaStream_t)stream);
}

int hsr_warp_src_row_range(const double* coords, int64_t rows, int64_t Wd, int64_t Hs, int64_t Ws,
                           const hsr_warp_geo_t* geo, int kernel, unsigned long long* range, void* stream) {
    return hsr::warp_src_row_range_impl(coords, rows, Wd, Hs, Ws, geo, kernel, range, (cudaStream_t)stream);
}

int hsr_warp_planes_window_f32(const float* src, int64_t Hs, int64_t Ws, int K, int64_t src_plane_stride,
                               const uint8_t* src_valid, int64_t src_row0, int64_t src_rows, const double* coords,
                               const hsr_warp_geo_t* geo, int kernel, const float* fill_out, int gate_k, float gate_gt,
                               int64_t Hd, int64_t Wd, float* dst, int64_t dst_plane_stride, uint8_t* dst_valid,
                               uint8_t* fit_mask, unsigned long long* outside, void* stream) {
    return hsr::warp_planes_window_impl(src, Hs, Ws, K, src_plane_stride, src_valid, src_row0, src_rows, coords, geo,
                                        kernel, fill_out, gate_k, gate_gt, Hd, Wd, dst, dst_plane_stride, dst_valid,
                                        fit_mask, outside, (cudaStream_t)stream);
}

int hsr_affine_fit_f64(const double* X, const double* Ybar, int64_t ns, int C, double* W, void* stream) {
    return hsr::affine_fit_impl(X, Ybar, ns, C, W, (cudaStream_t)stream);
}

int hsr_affine_apply_f32(const float* rgb, const double* W, const uint8_t* mask, int64_t n, int C, float lo, float hi,
                         float* out, void* stream) {
    return hsr::affine_apply_impl(rgb, W, mask, n, C, lo, hi, out, (cudaStream_t)stream);
}

int hsr_stretch_f64(const float* x, int64_t x_k_stride, int64_t x_g_stride, const double* lohi, const uint8_t* mask,
                    int64_t n, int K, int G, double* out, int64_t out_k_stride, int64_t out_g_stride, void* stream) {
    return hsr::stretch64_impl(x, x_k_stride, x_g_stride, lohi, mask, n, K, G, out, out_k_stride, out_g_stride,
                               (cudaStream_t)stream);
}

int hsr_notnan_mask_u8(const float* x, const uint8_t* base, int64_t n, uint8_t* out, void* stream) {
    return hsr::notnan_mask_impl(x, base, n, out, (cudaStream_t)stream);
}

int hsr_run_ends_u8(const float* sorted, int64_t n, uint8_t* flags, void* stream) {
    return hsr::run_ends_impl(sorted, n, flags, (cudaStream_t)stream);
}

int hsr_hist_match_f32(const float* src, const uint8_t* mask, int64_t n, const float* src_sorted, int64_t ns,
                       const float* ref_sorted, int64_t nr, const int32_t* ref_run_ends, int64_t nu, float* out, void* stream) {
    return hsr::hist_match_impl(src, mask, n, src_sorted, ns, ref_sorted, nr, ref_run_ends, nu, out, (cudaStream_t)stream);
}

size_t hsr_peer_block_bytes(void) { return hsr::peer_block_bytes(); }
int hsr_peer_alloc(void** dptr) { return hsr::peer_alloc_impl(dptr); }
int hsr_peer_free(void* dptr) { return hsr::peer_free_impl(dptr); }
int hsr_ipc_export(const void* dptr, unsigned char* handle) { return hsr::ipc_export_impl(dptr, handle); }
int hsr_ipc_import(const unsigned char* handle, void** dptr) { return hsr::ipc_import_impl(handle, dptr); }
int hsr_ipc_close(void* dptr) { return hsr::ipc_close_impl(dptr); }
int hsr_peer_status(const void* my_block, unsigned int* status, void* stream) {
    return hsr::peer_status_impl(my_block, status, (cudaStream_t)stream);
}
int hsr_allreduce_moments(double* moments, int64_t count, void* nccl_comm, void* stream) {
    return hsr::allreduce_moments_impl(moments, count, nccl_comm, (cudaStream_t)stream);
}

size_t hsr_workspace_bytes(int op, int64_t n, int K, int deg) {
    if (op == HSR_OP_POLY_MOMENTS) return hsr::poly_moments_workspace(n, K, deg);
    return 0;
}

}  // extern "C"
