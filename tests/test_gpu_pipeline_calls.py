"""The launch structure of every PairSynthesizer entry point: the C-ABI functions (``hsr_*``) each one calls, in order,
on small seeded inputs, against the sequences written down when the entry points were folded into one fit-and-apply
tail.  A change here means an entry point now launches differently: an extra mask or select, a lost fused path (the
y_finite mask inside the moment kernel, the one-pass percentile select of a single unit), or a moment sum or solve that
moved.  ``SCENARIOS`` is also the input set of profiles/pipetail/ab_results.py."""
import numpy as np
import pytest
import torch

from hsr_b200 import _lib, synthetic
from hsr_b200.EMIT_data import warp as hwarp
from hsr_b200.pipeline import PairSynthesizer, s2_target
from hsr_b200.s2_emit.srf import synthetic_s2_srf

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

GLT_GT = (-118.30, 0.000542232520256367, 0.0, 34.20, 0.0, -0.000542232520256367)
S2 = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3800040.0, dx=10.0, dy=10.0, width=10980, height=10980)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _ps(**kw):
    w = synthetic.emit_wavelengths()
    return PairSynthesizer(w, synthetic_s2_srf(), synthetic.good_band_mask(w), deg=2, device="cuda", **kw)


def _ref(K, shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand((K,) + tuple(shape), device="cuda", generator=g)


def _granule(ps, seed, Hr=40, Wr=34, on_grid=False):
    w = synthetic.emit_wavelengths()
    raw = synthetic.raw_cube_spectra_np((Hr, Wr, 285), seed=seed, good=synthetic.good_band_mask(w))
    raw[11, 9, 40] = np.nan
    gx, gy = synthetic.rotation_glt(Hr, Wr, 25.0)
    gx, gy = synthetic.inject_glt_defects(gx, gy, Hr, Wr, seed=seed + 1, hole_frac=0.01, n_oob=4, n_neg=4)
    g = {"raw": dev(raw), "glt_x": dev(gx), "glt_y": dev(gy)}
    shape = gx.shape
    if on_grid:
        g["target"] = s2_target(GLT_GT, gx.shape, S2)
        g["target"].coords(torch.device("cuda"))               # cached: the sequences hold no coordinate launch
        shape = g["target"].shape
    g["s2_ref"] = _ref(ps.K, shape, seed + 100)
    return g


def _synthesize(**kw):
    ps = _ps(**kw)
    g = _granule(ps, 0)
    return lambda: ps.synthesize(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"])


def _on_s2_grid():
    ps = _ps()
    g = _granule(ps, 1, on_grid=True)
    return lambda: ps.synthesize_on_s2_grid(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"], g["target"])


def _slab():
    ps = _ps()
    g = _granule(ps, 2)
    raw_host = g["raw"].cpu().pin_memory()
    r0, r1 = 10, 25
    return lambda: ps.synthesize_slab(raw_host, g["glt_x"][r0:r1], g["glt_y"][r0:r1], g["s2_ref"][:, r0:r1].contiguous())


def _slab_on_s2_grid():
    ps = _ps()
    g = _granule(ps, 3, on_grid=True)
    t = g["target"]
    Hd = t.shape[0]
    raw_host = g["raw"].cpu().pin_memory()
    rows = (Hd // 3, 2 * Hd // 3)
    return lambda: ps.synthesize_slab_on_s2_grid(raw_host, g["glt_x"], g["glt_y"],
                                                 g["s2_ref"][:, rows[0]:rows[1]].contiguous(), t, rows)


def _tiles(**kw):
    ps = _ps(min_count=50, **kw)
    w = synthetic.emit_wavelengths()
    T, h = 3, 24
    raws = np.stack([synthetic.raw_cube_spectra_np((h, h, 285), seed=20 + t, good=synthetic.good_band_mask(w))
                     for t in range(T)])
    glts = [synthetic.identity_glt(h, h, 0.02, seed=2 + t) for t in range(T)]
    gx, gy = np.stack([g[0] for g in glts]), np.stack([g[1] for g in glts])
    s2 = _ref(ps.K, (T, h, h), 7)
    return lambda: ps.synthesize_tiles(dev(raws), dev(gx), dev(gy), s2)


def _sharded(n, **kw):
    ps = _ps(**kw)
    gs = [_granule(ps, 30 + i, Hr=30 + 4 * i, on_grid=(i == 2)) for i in range(n)]
    return lambda: ps.synthesize_sharded(gs)


def _fine():
    ps = _ps(stretch=(2, 98))
    g = _granule(ps, 5)
    res = ps.synthesize(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"])
    return lambda: ps.matched_fine(res, 3)


FIT = {"stretch": (2, 98), "stretch_scope": "fit"}
OT = {"targets": "ot", "n_samples": 300}
SCENARIOS = {
    "synthesize": lambda: _synthesize(),
    "synthesize_y_finite": lambda: _synthesize(y_finite=True),
    "synthesize_stretch": lambda: _synthesize(stretch=(2, 98)),
    "synthesize_stretch_y_finite": lambda: _synthesize(stretch=(2, 98), y_finite=True),
    "synthesize_on_s2_grid": _on_s2_grid,
    "synthesize_slab": _slab,
    "synthesize_slab_on_s2_grid": _slab_on_s2_grid,
    "synthesize_tiles": lambda: _tiles(),
    "synthesize_tiles_stretch_y_finite": lambda: _tiles(stretch=(2, 98), y_finite=True),
    "sharded_0": lambda: _sharded(0),
    "sharded_1": lambda: _sharded(1),
    "sharded_3": lambda: _sharded(3),
    "sharded_0_fit": lambda: _sharded(0, **FIT),
    "sharded_1_fit": lambda: _sharded(1, **FIT),
    "sharded_3_fit": lambda: _sharded(3, **FIT),
    "sharded_3_y_finite": lambda: _sharded(3, y_finite=True),
    "sharded_3_fit_y_finite": lambda: _sharded(3, y_finite=True, **FIT),
    "synthesize_ot": lambda: _synthesize(**OT),
    "synthesize_ot_stretch_y_finite": lambda: _synthesize(stretch=(2, 98), y_finite=True, **OT),
    "sharded_3_ot": lambda: _sharded(3, **OT),
    "sharded_3_ot_y_finite": lambda: _sharded(3, y_finite=True, **OT),
    "sharded_3_ot_fit_y_finite": lambda: _sharded(3, y_finite=True, **FIT, **OT),
    "matched_fine": _fine,
}

# Recorded from the entry points before they shared one tail, with two changes, both on the sharded OT path with
# y_finite: each granule's fit mask is taken once, right after its planes, as the paired path does.  With a stretch
# the second mask launch per granule is gone; without one the same launches moved from after every granule's planes.
EXPECTED = {
    "matched_fine":
        "bilinear_fine_mask_u8 union_select_state_bytes union_select_hist_doubles union_select_begin "
        "union_select_count_bilinear union_select_step union_select_count_bilinear union_select_step "
        "union_select_count_bilinear union_select_step union_select_count_bilinear union_select_step "
        "bilinear_apply_f32",
    "sharded_0": "moments_sum_f64",
    "sharded_0_fit":
        "union_select_state_bytes union_select_hist_doubles union_select_begin union_select_step "
        "union_select_step union_select_step union_select_step moments_sum_f64",
    "sharded_1": "glt_srf_f32 fit_moments_workspace_bytes fit_moments_f64 moments_sum_f64 poly_solve_apply_f32",
    "sharded_1_fit":
        "glt_srf_f32 percentiles_workspace_bytes masked_percentiles_pair_f64 fit_moments_workspace_bytes "
        "fit_moments_f64 moments_sum_f64 poly_solve_apply_f32",
    "sharded_3":
        "glt_srf_f32 glt_srf_f32 glt_srf_f32 warp_planes_f32 fit_moments_workspace_bytes fit_moments_f64 "
        "fit_moments_workspace_bytes fit_moments_f64 fit_moments_workspace_bytes fit_moments_f64 "
        "moments_sum_f64 poly_solve_apply_f32 poly_solve_apply_f32 poly_solve_apply_f32",
    "sharded_3_fit":
        "glt_srf_f32 glt_srf_f32 glt_srf_f32 warp_planes_f32 union_select_state_bytes union_select_hist_doubles "
        "union_select_begin union_select_count union_select_count union_select_count union_select_step "
        "union_select_count union_select_count union_select_count union_select_step union_select_count "
        "union_select_count union_select_count union_select_step union_select_count union_select_count "
        "union_select_count union_select_step fit_moments_workspace_bytes fit_moments_f64 "
        "fit_moments_workspace_bytes fit_moments_f64 fit_moments_workspace_bytes fit_moments_f64 "
        "moments_sum_f64 poly_solve_apply_f32 poly_solve_apply_f32 poly_solve_apply_f32",
    "sharded_3_fit_y_finite":
        "glt_srf_f32 fit_mask_u8 glt_srf_f32 fit_mask_u8 glt_srf_f32 warp_planes_f32 fit_mask_u8 "
        "union_select_state_bytes union_select_hist_doubles union_select_begin union_select_count "
        "union_select_count union_select_count union_select_step union_select_count union_select_count "
        "union_select_count union_select_step union_select_count union_select_count union_select_count "
        "union_select_step union_select_count union_select_count union_select_count union_select_step "
        "fit_moments_workspace_bytes fit_moments_f64 fit_moments_workspace_bytes fit_moments_f64 "
        "fit_moments_workspace_bytes fit_moments_f64 moments_sum_f64 poly_solve_apply_f32 poly_solve_apply_f32 "
        "poly_solve_apply_f32",
    "sharded_3_ot":
        "glt_srf_f32 glt_srf_f32 glt_srf_f32 warp_planes_f32 compact_planes_pair_workspace_bytes "
        "compact_planes_pair compact_planes_pair_workspace_bytes compact_planes_pair "
        "compact_planes_pair_workspace_bytes compact_planes_pair gather_planes_f64 gather_planes_f64 "
        "gather_planes_f64 gather_planes_f64 gather_planes_f64 gather_planes_f64 sinkhorn_workspace_bytes "
        "sinkhorn_barycentric_k_f64 polyfit_moments_f64in poly_solve_apply_f32 poly_solve_apply_f32 "
        "poly_solve_apply_f32",
    "sharded_3_ot_fit_y_finite":
        "glt_srf_f32 fit_mask_u8 glt_srf_f32 fit_mask_u8 glt_srf_f32 warp_planes_f32 fit_mask_u8 "
        "union_select_state_bytes union_select_hist_doubles union_select_begin union_select_count "
        "union_select_count union_select_count union_select_step union_select_count union_select_count "
        "union_select_count union_select_step union_select_count union_select_count union_select_count "
        "union_select_step union_select_count union_select_count union_select_count union_select_step "
        "compact_planes_pair_workspace_bytes compact_planes_pair compact_planes_pair_workspace_bytes "
        "compact_planes_pair compact_planes_pair_workspace_bytes compact_planes_pair gather_planes_f64 "
        "gather_planes_f64 gather_planes_f64 gather_planes_f64 gather_planes_f64 gather_planes_f64 "
        "sinkhorn_workspace_bytes sinkhorn_barycentric_k_f64 polyfit_moments_f64in poly_solve_apply_f32 "
        "poly_solve_apply_f32 poly_solve_apply_f32",
    "sharded_3_ot_y_finite":
        "glt_srf_f32 fit_mask_u8 glt_srf_f32 fit_mask_u8 glt_srf_f32 warp_planes_f32 fit_mask_u8 "
        "compact_planes_pair_workspace_bytes compact_planes_pair compact_planes_pair_workspace_bytes "
        "compact_planes_pair compact_planes_pair_workspace_bytes compact_planes_pair gather_planes_f64 "
        "gather_planes_f64 gather_planes_f64 gather_planes_f64 gather_planes_f64 gather_planes_f64 "
        "sinkhorn_workspace_bytes sinkhorn_barycentric_k_f64 polyfit_moments_f64in poly_solve_apply_f32 "
        "poly_solve_apply_f32 poly_solve_apply_f32",
    "sharded_3_y_finite":
        "glt_srf_f32 glt_srf_f32 glt_srf_f32 warp_planes_f32 fit_moments_workspace_bytes fit_moments_f64 "
        "fit_moments_workspace_bytes fit_moments_f64 fit_moments_workspace_bytes fit_moments_f64 "
        "moments_sum_f64 poly_solve_apply_f32 poly_solve_apply_f32 poly_solve_apply_f32",
    "synthesize": "glt_srf_f32 fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_on_s2_grid":
        "glt_srf_f32 warp_planes_f32 fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_ot":
        "glt_srf_f32 compact_planes_pair_workspace_bytes compact_planes_pair gather_planes_f64 "
        "gather_planes_f64 sinkhorn_workspace_bytes sinkhorn_barycentric_k_f64 polyfit_moments_f64in "
        "poly_solve_apply_f32",
    "synthesize_ot_stretch_y_finite":
        "glt_srf_f32 fit_mask_u8 percentiles_workspace_bytes masked_percentiles_pair_f64 "
        "compact_planes_pair_workspace_bytes compact_planes_pair gather_planes_f64 gather_planes_f64 "
        "sinkhorn_workspace_bytes sinkhorn_barycentric_k_f64 polyfit_moments_f64in poly_solve_apply_f32",
    "synthesize_slab": "glt_row_range glt_srf_f32 fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_slab_on_s2_grid":
        "warp_coords_rows_f64 warp_src_row_range glt_row_range glt_srf_f32 warp_planes_window_f32 "
        "fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_stretch":
        "glt_srf_f32 percentiles_workspace_bytes masked_percentiles_pair_f64 fit_moments_workspace_bytes "
        "fit_moments_f64 poly_solve_apply_f32",
    "synthesize_stretch_y_finite":
        "glt_srf_f32 fit_mask_u8 percentiles_workspace_bytes masked_percentiles_pair_f64 "
        "fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_tiles": "glt_srf_f32 fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_tiles_stretch_y_finite":
        "glt_srf_f32 fit_mask_u8 percentiles_workspace_bytes masked_percentiles_pair_f64 "
        "fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
    "synthesize_y_finite": "glt_srf_f32 fit_moments_workspace_bytes fit_moments_f64 poly_solve_apply_f32",
}


class _Recorder:
    """Stands in for the loaded library: forwards every call and records the name of each ``hsr_*`` function."""

    def __init__(self, handle):
        self._handle, self.calls = handle, []

    def __getattr__(self, name):
        fn = getattr(self._handle, name)
        if not name.startswith("hsr_"):
            return fn

        def call(*args):
            self.calls.append(name[4:])
            return fn(*args)
        return call


def run_recorded(name):
    """``(result, names of the hsr_* calls)`` of scenario ``name``; the inputs are built before the recording starts."""
    run = SCENARIOS[name]()
    real = _lib.lib
    rec = _Recorder(real())
    _lib.lib = lambda: rec
    try:
        out = run()
        torch.cuda.synchronize()
    finally:
        _lib.lib = real
    return out, " ".join(rec.calls)


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_launch_sequence(name):
    assert run_recorded(name)[1] == EXPECTED[name]
