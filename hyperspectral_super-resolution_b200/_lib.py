"""ctypes binding of ``csrc/libhsr_b200.so`` (C ABI: ``include/hsr_b200.h``).

The library is built in-tree by :func:`build` (``make`` -> nvcc, sm_100a only).  Loading is
lazy; :func:`lib` raises ``HsrLibraryError`` when the shared object is missing — there is no
other implementation to fall back to.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC_DIR, "libhsr_b200.so")
ABI_VERSION = 7
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "hsr_b200.h")

HSR_OP_POLY_MOMENTS = 1
HSR_FIT_MASK_GIVEN = 1
HSR_FIT_Y_FINITE = 2
HSR_MAX_SRF_BANDS = 16
HSR_MAX_POLY_DEG = 8
HSR_TILE_PX = 32
HSR_MAX_PERCENTILES = 2
HSR_PEER_TIMEOUT = 1
HSR_EPEER = -5
HSR_ENCCL = -6


class Exchange(ctypes.Structure):
    """hsr_exchange_t of include/hsr_b200.h."""
    _fields_ = [("peer_blocks", ctypes.c_void_p), ("my_block", ctypes.c_void_p), ("nranks", ctypes.c_int),
                ("rank", ctypes.c_int), ("epoch", ctypes.c_ulonglong), ("timeout_ms", ctypes.c_uint),
                ("reserved", ctypes.c_uint)]


class RawView(ctypes.Structure):
    """hsr_raw_view_t of include/hsr_b200.h."""
    _fields_ = [("row0", ctypes.c_int64), ("rows", ctypes.c_int64), ("batch_out_rows", ctypes.c_int64),
                ("batch_raw_rows", ctypes.c_int64)]


class WarpGeo(ctypes.Structure):
    """hsr_warp_geo_t of include/hsr_b200.h."""
    _fields_ = [("src_gt", ctypes.c_double * 6), ("dst_gt", ctypes.c_double * 6), ("utm_zone", ctypes.c_int),
                ("south", ctypes.c_int), ("xscale", ctypes.c_double), ("yscale", ctypes.c_double)]


class HsrLibraryError(RuntimeError):
    """libhsr_b200.so is missing or could not be loaded."""


class HsrError(RuntimeError):
    """A C-ABI call returned non-zero (``code`` < 0: argument error, > 0: cudaError_t)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"hsr_b200 error {code}: {message}")
        self.code = code


_c = ctypes
_p = _c.c_void_p
_i64 = _c.c_int64
_int = _c.c_int
_f32 = _c.c_float

# name -> (restype, argtypes); mirrors include/hsr_b200.h one to one
SIGNATURES = {
    "hsr_version": (_int, []),
    "hsr_last_error": (_c.c_char_p, []),
    "hsr_glt_ortho_f32": (_int, [_p, _i64, _i64, _int, _i64, _int, _p, _p, _i64, _i64, _i64, _f32,
                                 _p, _i64, _p, _p, _p, _p]),
    "hsr_glt_srf_f32": (_int, [_p, _i64, _i64, _int, _i64, _int, _p, _p, _i64, _i64, _i64, _f32,
                               _p, _p, _int, _p, _i64, _p, _i64, _p, _p, _p, _int, _f32, _p, _p]),
    "hsr_glt_ortho_u16": (_int, [_p, _i64, _i64, _int, _i64, _int, _p, _p, _i64, _i64, _i64, _f32, _f32, _int, _f32, _int,
                                 _p, _i64, _p, _p, _f32, _f32, _f32, _f32, _p, _p, _p]),
    "hsr_glt_row_range": (_int, [_p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p]),
    "hsr_srf_f32": (_int, [_p, _i64, _int, _i64, _p, _int, _p, _i64, _p, _int, _f32, _p]),
    "hsr_poly_moments_f64": (_int, [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _i64, _i64, _int, _int, _p, _p, _p]),
    "hsr_poly_solve_f64": (_int, [_p, _int, _int, _i64, _p, _p]),
    "hsr_poly_apply_f32": (_int, [_p, _i64, _i64, _p, _p, _i64, _i64, _i64, _int, _int, _f32, _f32,
                                  _p, _i64, _i64, _p]),
    "hsr_fit_mask_u8": (_int, [_p, _i64, _i64, _p, _i64, _i64, _i64, _int, _int, _p, _int, _f32, _p, _p]),
    "hsr_fit_moments_f64": (_int, [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _int, _int, _f32,
                                   _int, _p, _p, _p, _p, _p, _p, _p]),
    "hsr_fit_moments_workspace_bytes": (_c.c_size_t, [_i64, _int, _int, _int]),
    "hsr_poly_solve_apply_f32": (_int, [_p, _i64, _i64, _p, _p, _i64, _int, _int, _int, _i64, _f32, _f32, _p, _p,
                                        _p, _i64, _i64, _p, _p, _p]),
    "hsr_block_average_f32": (_int, [_p, _int, _int, _i64, _i64, _i64, _int, _int, _c.c_double, _int, _f32, _p, _i64, _p]),
    "hsr_bilinear_upsample_f32": (_int, [_p, _int, _i64, _i64, _i64, _int, _int, _f32, _p, _i64, _p]),
    "hsr_stretch_f64": (_int, [_p, _i64, _i64, _p, _p, _i64, _int, _int, _p, _i64, _i64, _p]),
    "hsr_notnan_mask_u8": (_int, [_p, _p, _i64, _p, _p]),
    "hsr_run_ends_u8": (_int, [_p, _i64, _p, _p]),
    "hsr_hist_match_f32": (_int, [_p, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p]),
    "hsr_affine_fit_f64": (_int, [_p, _p, _i64, _int, _p, _p]),
    "hsr_affine_apply_f32": (_int, [_p, _p, _p, _i64, _int, _f32, _f32, _p, _p]),
    "hsr_warp_f32": (_int, [_p, _i64, _i64, _int, _i64, _p, _int, _int, _f32, _f32, _i64, _i64, _p, _i64, _p, _c.c_size_t,
                            _p]),
    "hsr_warp_workspace_bytes": (_c.c_size_t, [_i64, _i64]),
    "hsr_warp_coords_f64": (_int, [_p, _i64, _i64, _p, _p]),
    "hsr_warp_planes_f32": (_int, [_p, _i64, _i64, _int, _i64, _p, _p, _p, _int, _p, _int, _f32, _i64, _i64, _p, _i64,
                                   _p, _p, _p]),
    "hsr_peer_block_bytes": (_c.c_size_t, []),
    "hsr_peer_alloc": (_int, [_p]),
    "hsr_peer_free": (_int, [_p]),
    "hsr_ipc_export": (_int, [_p, _p]),
    "hsr_ipc_import": (_int, [_p, _p]),
    "hsr_ipc_close": (_int, [_p]),
    "hsr_peer_status": (_int, [_p, _p, _p]),
    "hsr_allreduce_moments": (_int, [_p, _i64, _p, _p]),
    "hsr_moments_sum_f64": (_int, [_p, _int, _i64, _p, _p, _p]),
    "hsr_workspace_bytes": (_c.c_size_t, [_int, _i64, _int, _int]),
    "hsr_compact_workspace_bytes": (_c.c_size_t, [_i64]),
    "hsr_compact_finite_rows": (_int, [_p, _p, _i64, _int, _p, _p, _p, _p]),
    "hsr_gather_rows_f64": (_int, [_p, _p, _p, _i64, _int, _p, _p]),
    "hsr_sinkhorn_workspace_bytes": (_c.c_size_t, [_int, _int]),
    "hsr_sinkhorn_barycentric_f64": (_int, [_p, _p, _int, _int, _int, _c.c_double, _int, _c.c_double, _p, _p, _p, _p]),
    "hsr_polyfit_moments_f64in": (_int, [_p, _p, _i64, _int, _int, _p, _p]),
    "hsr_black_mask_f32": (_int, [_p, _i64, _i64, _i64, _int, _int, _int, _f32, _f32, _f32, _f32, _f32, _p, _p, _p]),
    "hsr_quantize_u16_f32": (_int, [_p, _i64, _int, _f32, _f32, _int, _p, _p]),
    "hsr_tile_sums_u8": (_int, [_p, _i64, _i64, _int, _int, _int, _int, _p, _p]),
    "hsr_percentiles_workspace_bytes": (_c.c_size_t, [_i64, _int, _int, _int]),
    "hsr_masked_percentiles_pair_f64": (_int, [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _int, _int, _p, _int, _p, _p, _p, _p]),
    "hsr_masked_percentiles_f64": (_int, [_p, _i64, _i64, _p, _i64, _int, _int, _p, _int, _p, _p, _p]),
    "hsr_stretch_f32": (_int, [_p, _i64, _i64, _p, _i64, _int, _int, _p, _i64, _i64, _p]),
    "hsr_union_select_state_bytes": (_c.c_size_t, [_int, _int]),
    "hsr_union_select_hist_doubles": (_i64, [_int, _int]),
    "hsr_union_select_begin": (_int, [_p, _int, _int, _p, _p, _p]),
    "hsr_union_select_count": (_int, [_p, _i64, _p, _i64, _p, _i64, _int, _int, _int, _p, _p, _p]),
    "hsr_union_select_step": (_int, [_int, _int, _int, _p, _p, _p, _p, _p]),
}

_lock = threading.Lock()
_handle = None


def build(verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a into ``csrc/libhsr_b200.so`` (nvcc cross-compiles without a GPU)."""
    proc = subprocess.run(["make", "-C", CSRC_DIR, "-j8"], capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        print(proc.stdout)
        print(proc.stderr)
    if proc.returncode != 0:
        raise HsrLibraryError(f"building libhsr_b200.so failed (exit {proc.returncode})")
    return LIB_PATH


def lib() -> ctypes.CDLL:
    """Return the loaded library, loading it on first use."""
    global _handle
    if _handle is not None:
        return _handle
    with _lock:
        if _handle is None:
            path = LIB_PATH  # the module global, read at call time
            if not os.path.exists(path):
                raise HsrLibraryError(
                    f"{path} not found — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    f"or `make -C {CSRC_DIR}`; hsr_b200 has no CPU fallback")
            try:
                h = ctypes.CDLL(path)
            except OSError as e:  # pragma: no cover
                raise HsrLibraryError(f"cannot load {path}: {e}") from e
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(h, name)
                fn.restype = res
                fn.argtypes = args
            if h.hsr_version() != ABI_VERSION:
                raise HsrLibraryError(f"{path} has ABI version {h.hsr_version()}, this package needs {ABI_VERSION}: "
                                      "rebuild it (python -c 'import __graft_entry__ as g; g.build()')")
            _handle = h
    return _handle


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().hsr_last_error()
        raise HsrError(rc, msg.decode("utf-8", "replace") if msg else "unknown error")
