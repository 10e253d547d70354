"""The C-ABI library loads and exports every symbol include/hsr_b200.h declares (no compute calls:
there is no GPU in the build container)."""
import ctypes
import os
import re

import pytest

from hsr_b200 import _lib


def _declared_symbols():
    text = open(_lib.HEADER_PATH).read()
    return sorted(set(re.findall(r"HSR_API\s+[\w\s\*]+?\b(hsr_\w+)\s*\(", text)))


def test_header_declares_the_hot_path():
    names = _declared_symbols()
    for must in ("hsr_glt_ortho_f32", "hsr_glt_srf_f32", "hsr_srf_f32", "hsr_poly_moments_f64",
                 "hsr_poly_solve_f64", "hsr_poly_apply_f32", "hsr_fit_mask_u8", "hsr_workspace_bytes",
                 "hsr_version", "hsr_last_error"):
        assert must in names


def test_library_exports_every_declared_symbol():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    h = ctypes.CDLL(_lib.LIB_PATH)
    for name in _declared_symbols():
        assert hasattr(h, name), f"{name} declared in hsr_b200.h but not exported by libhsr_b200.so"


def test_binding_table_covers_header_one_to_one():
    assert sorted(_lib.SIGNATURES) == _declared_symbols()


def test_abi_v7_version_and_workspace_are_callable_without_a_gpu():
    lib = _lib.lib()
    assert lib.hsr_version() == 7
    ws = lib.hsr_workspace_bytes(_lib.HSR_OP_POLY_MOMENTS, 1685 * 1667, 12, 2)
    assert ws > 0 and ws % (12 * 8 * 8) == 0
    assert lib.hsr_workspace_bytes(99, 10, 1, 2) == 0
    assert lib.hsr_workspace_bytes(_lib.HSR_OP_POLY_MOMENTS, 10, 1, 99) == 0


def test_header_limits_match_python_constants():
    text = open(_lib.HEADER_PATH).read()
    assert int(re.search(r"#define HSR_MAX_SRF_BANDS (\d+)", text).group(1)) == _lib.HSR_MAX_SRF_BANDS
    assert int(re.search(r"#define HSR_MAX_POLY_DEG (\d+)", text).group(1)) == _lib.HSR_MAX_POLY_DEG
    assert int(re.search(r"#define HSR_TILE_PX (\d+)", text).group(1)) == _lib.HSR_TILE_PX


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(_lib, "_handle", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.HsrLibraryError):
        _lib.lib()


def test_product_library_reads_no_environment_variable():
    """VERDICT r1: work-skipping / tuning knobs must not ship.  The library has no getenv at all, and none of the knob
    names INTEGRATION.md lists appears in it."""
    import subprocess

    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    und = subprocess.run(["nm", "-D", "--undefined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = {ln.split()[-1].split("@")[0] for ln in und.splitlines() if ln.strip()}
    assert "getenv" not in names and "secure_getenv" not in names
    strings = subprocess.run(["strings", "-n", "6", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    knobs = ("HSR_DRY_CONSUMER", "HSR_WARP_DRY", "HSR_STAGES", "HSR_PRODUCERS", "HSR_NO_MERGE", "HSR_GLT_NO_RING",
             "HSR_GLT_BULK", "HSR_L2_STREAM", "HSR_FIT_REVERSE", "HSR_OT_UNFUSED", "HSR_OT_NO_GRAPH", "HSR_WARP_NO_QUAD",
             "HSR_WARP_NO_LANE", "HSR_Q16_PAIR")
    assert [k for k in knobs if k in strings] == []


def test_exchange_descriptor_must_alternate_fit_then_solve():
    """ADVICE r1: a peer-exchange descriptor goes through fit_moments (stage 1) then poly_solve_apply (stage 2),
    once each; anything else raises on the host instead of dead-locking the device."""
    from hsr_b200 import kernels

    ex = _lib.Exchange(0, 0, 2, 0, 0, 0, 0)
    ex._stage = 0
    with pytest.raises(RuntimeError, match="out of order"):
        kernels._exchange_arg(ex, 2)                      # solve before fit
    assert kernels._exchange_arg(ex, 1) is not None
    with pytest.raises(RuntimeError, match="out of order"):
        kernels._exchange_arg(ex, 1)                      # second fit on the same descriptor
    assert kernels._exchange_arg(ex, 2) is not None
    assert kernels._exchange_arg(None, 1) is None
    assert ctypes.sizeof(_lib.Exchange) == 40             # hsr_exchange_t: 2 pointers, 2 ints, u64, 2 u32
