"""The pair-synthesis pass: GLT ortho + SRF bands + per-band polynomial colour matching.

This is the composition the reference spreads over ``nc_to_envi`` (emit_proj.py:968-987), a disk
round trip, ``pseudo_s2_srf_integral`` (synth.py:9-45) and the fit / apply of
``poly_regression.py:104-139`` — here three kernel launches (plus a tiny fixed-order finalize) on one stream, the raw cube read
from HBM once:

    glt_srf          raw cube + GLT  -> K pseudo-S2 planes, valid mask, diag AND the fit mask (valid & finite &
                     first band > 0, poly_regression.py:106) while the planes are written; optional ortho cube
    fit_moments      fp64 normal equations of the planes vs the S2 reference under that mask
                     [+ all-reduce across ranks]
    poly_solve_apply (K, deg+1) coefficients and the colour-matched planes, clipped to [0, 1]

``synthesize_on_s2_grid`` runs the same pass on the Sentinel-2 UTM grid, where the reference fits: glt_srf, then a warp
of the K planes onto the S2 grid (``warp_planes``), then the same fit and solve / apply.  ``synthesize_sharded`` takes
granules with an S2 target too, and ``synthesize_slab_on_s2_grid`` runs one band of target rows of a mosaic, staging only
the ortho and raw rows that band reads.

``targets="ot"`` fits the polynomial against the optimal-transport barycentric targets of the reference script
(poly_regression.py:129-137, ``fit_ot_poly_rgb``) instead of the pixel-paired ones: a planar compaction of the fit
mask, the sample draw on the host, a planar gather, the fp64 Sinkhorn and the moments of (X, Ybar) feeding the same
solve / apply (``_ot_moments``; DESIGN section 4.9).

Every ``synthesize*`` entry point produces its planes and masks as units and hands them to one fit-and-apply tail
(``_fit_apply``).

``matched_fine`` takes a result to the Sentinel-2 10 m resolution as the reference script's last step does
(poly_regression.py:150-162): bilinear x factor of the planes, mask, the stretch with the percentiles of the fine planes
and the 60 m polynomial — a fine mask, a union select over the fine values computed on the fly, and one fused apply.
"""
from __future__ import annotations

from dataclasses import dataclass, replace
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np
import torch

from . import dist as hdist
from . import kernels
from ._host import cuda_device, to_device
from .EMIT_data.warp import S2Target, s2_target, warp_planes  # noqa: F401  (the building blocks of synthesize_on_s2_grid)
from .s2_emit.srf import srf_fold_weights

NO_DATA_VALUE = kernels.NO_DATA_VALUE
STRETCH_SCOPES = ("granule", "fit")
TARGETS = ("paired", "ot")


def _no_reduce(t):
    return t


@dataclass
class PairResult:
    bands: torch.Tensor                 # [K, Ho, Wo] f32 pseudo-S2 planes (x of the fit)
    matched: torch.Tensor               # [K, Ho, Wo] f32 colour-matched planes
    coeffs: torch.Tensor                # [K, deg+1] (or [K, T, deg+1] for tile batches) f64
    valid: torch.Tensor                 # [Ho, Wo] bool: GLT entry valid and in bounds
    fit_mask: torch.Tensor              # [Ho, Wo] bool: pixels that entered the fit / were mapped
    diag: torch.Tensor                  # int64[3] GLT diagnostics (device)
    moments: torch.Tensor               # [K, 3*deg+2] f64 (after the all-reduce, if any)
    ortho: Optional[torch.Tensor] = None    # [Ho, Wo, B] f32 when materialised
    band_names: Optional[List[str]] = None
    x_limits: Optional[torch.Tensor] = None  # [K, G, 2] f64 (lo, hi) percentile stretch of the planes, if enabled
                                             # ([K, 1, 2], the same on every rank, for a global fit with stretch_scope="fit")
    y_limits: Optional[torch.Tensor] = None  # ... and of the S2 reference
    raw_rows: Optional[tuple] = None         # synthesize_slab: the [row0, row1) raw rows that were staged
    grid: Optional[S2Target] = None          # synthesize_on_s2_grid: the S2 grid of bands / matched / valid / fit_mask
    ortho_rows: Optional[tuple] = None       # synthesize_slab_on_s2_grid: the [row0, row1) ortho rows that were staged
    ot_info: Optional[tuple] = None          # targets="ot": (iterations, err, err_iteration, numerical) of the Sinkhorn
                                             # (fit_ot_poly_rgb's return_info); None for paired fits and the identity


@dataclass
class FineResult:
    matched: torch.Tensor                    # [K, f*H, f*W] f32 colour-matched planes on the finer grid (padded planes)
    mask: torch.Tensor                       # [f*H, f*W] bool: mask10, every fine value finite
    x_limits: Optional[torch.Tensor]         # [K, 1, 2] f64 (lo, hi) percentiles of the fine planes, None without a stretch
    factor: int
    s2_window: Optional[tuple] = None        # the target's s2_window x factor: (row, col) of the top-left fine pixel in
                                             # the S2 grid at the fine resolution (None off the S2 grid)


@dataclass
class _Unit:
    """One image of a fit, as an entry point produced it: the fields of its PairResult before the fit."""
    bands: torch.Tensor                 # [K, Ho, Wo] (tile batches: [K, T, h, w]) f32 planes
    s2_ref: torch.Tensor
    valid: torch.Tensor                 # shaped as the result's valid / fit_mask
    fit_mask: torch.Tensor              # from glt_srf / warp_planes
    diag: torch.Tensor
    ortho: Optional[torch.Tensor] = None
    grid: Optional[S2Target] = None
    matched_out: Optional[torch.Tensor] = None


class PairSynthesizer:
    """Holds the folded SRF weights on the device and runs the fused pass for granules or tile batches."""

    def __init__(self, emit_w, srf_dict: Dict[str, tuple], good_mask=None, *, deg: int = 2,
                 fill: float = NO_DATA_VALUE, min_count: int = 200, gate_band: Optional[str] = None,
                 clip=(0.0, 1.0), y_finite: bool = False, stretch=None, stretch_scope: str = "granule", device=None,
                 targets: str = "paired", n_samples: int = 5000, reg: float = 0.05, numItermax: int = 300,
                 stopThr: float = 1e-6, seed=0):
        """``stretch=(pmin, pmax)`` inserts the shared percentile stretch of s2_emit/color.py:25-34 between the
        SRF synthesis and the fit, as the reference's script does (poly_regression.py:126-127): both images are
        stretched with their own masked percentiles, the fit and the apply then run on the stretched values
        (applied on the fly; the stretched planes are never written).

        ``stretch_scope`` says over which pixels the percentiles are taken.  "granule" (default): per image, and a
        global fit (``synthesize_sharded``, ``exchange=`` / ``allreduce=True``) with a stretch raises ``ValueError``.
        "fit": over exactly the pixels the fit is taken over — one granule, each tile of ``synthesize_tiles``, or the
        union of every granule / slab on every rank of a global fit (exact: np.percentile of the concatenation, the
        same limits on every rank).

        ``targets``: "paired" (default) fits every masked pixel against the reference at that pixel; "ot" fits against
        the optimal-transport barycentric targets of ``fit_ot_poly_rgb`` (poly_regression.py:129-137) with its
        ``n_samples``, ``reg``, ``numItermax``, ``stopThr`` and ``seed``, jointly over the K planes: X rows (all K planes
        finite, after the stretch if any) and Y rows (likewise) of the fit mask, the identity when either count is
        below ``min_count``, else ``default_rng(seed).choice`` samples of each, the fp64 Sinkhorn and the per-plane
        polynomial of X against the targets.  A global fit (``synthesize_sharded``, ``allreduce=True``) is that fit
        over the concatenation of every unit's rows in (rank, unit) order.  ``exchange=``, ``synthesize_tiles`` and
        ``HostGranuleStream`` raise ``ValueError`` with "ot" (DESIGN section 4.9)."""
        if stretch_scope not in STRETCH_SCOPES:
            raise ValueError(f"stretch_scope must be one of {STRETCH_SCOPES}, got {stretch_scope!r}")
        self.device = torch.device(device) if device is not None else cuda_device()
        W, names, none_bands, fill_out = srf_fold_weights(emit_w, srf_dict, good_mask, fill=fill)
        if not names:
            raise ValueError("no S2 band has a non-zero response on the EMIT grid")
        self.band_names, self.none_bands = names, none_bands
        self.W = to_device(W, torch.float32, self.device)
        self.fill_out = to_device(fill_out, torch.float32, self.device)
        self.deg, self.fill, self.min_count = int(deg), float(fill), int(min_count)
        if gate_band is not None and gate_band not in names:
            raise KeyError(f"gate_band {gate_band!r} is not among the synthesised bands {names}")
        self.gate_k = names.index(gate_band) if gate_band is not None else 0
        self.clip = clip
        self.y_finite = bool(y_finite)
        self.stretch = None if stretch is None else (float(stretch[0]), float(stretch[1]))
        self.stretch_scope = stretch_scope
        if targets not in TARGETS:
            raise ValueError(f"targets must be one of {TARGETS}, got {targets!r}")
        self.targets = targets
        if targets == "ot":
            if int(n_samples) != n_samples or n_samples < 1:
                raise ValueError(f"n_samples must be an integer >= 1, got {n_samples!r}")
            if not (float(reg) > 0.0 and np.isfinite(reg)):
                raise ValueError(f"reg must be a finite number > 0, got {reg!r}")
            if int(numItermax) != numItermax or numItermax < 0:
                raise ValueError(f"numItermax must be an integer >= 0, got {numItermax!r}")
            if np.isnan(float(stopThr)):
                raise ValueError("stopThr must not be NaN")
            try:
                np.random.default_rng(seed)
            except (TypeError, ValueError) as e:
                raise ValueError(f"seed {seed!r} is not a valid numpy.random.default_rng seed: {e}") from None
        self.n_samples, self.reg, self.numItermax = int(n_samples), float(reg), int(numItermax)
        self.stopThr, self.seed = float(stopThr), seed

    @property
    def K(self) -> int:
        return len(self.band_names)

    # ------------------------------------------------------------------ stage helpers
    def bands_from_raw(self, raw, glt_x, glt_y, *, transpose_raw_yx=False, materialize_ortho=False,
                       bands_out=None, ortho_out=None, fit_mask_out=None, raw_row0=0, raw_rows_total=None,
                       tile_rows=None, valid_out=None, want_diag=True):
        """(bands, valid, diag, ortho); with ``fit_mask_out`` ([Ho, Wo] bool) the kernel also writes the fit mask.
        ``raw_row0`` / ``raw_rows_total`` / ``tile_rows``: see :func:`hsr_b200.kernels.glt_ortho` (hsr_raw_view_t)."""
        return kernels.glt_srf(raw, glt_x, glt_y, self.W, self.fill_out, fill=self.fill,
                               transpose_raw_yx=transpose_raw_yx, materialize_ortho=materialize_ortho,
                               bands_out=bands_out, ortho_out=ortho_out, fit_mask_out=fit_mask_out,
                               gate_k=self.gate_k, gate_gt=0.0, raw_row0=raw_row0, raw_rows_total=raw_rows_total,
                               tile_rows=tile_rows, valid_out=valid_out, want_diag=want_diag)

    def fit(self, bands, s2_ref, valid, fit_mask, *, groups=1, exchange=None, reduce=None):
        """Moments under the fit mask the SRF kernel produced; with ``y_finite`` the mask is rebuilt from the
        planes so that non-finite reference pixels drop out of it as well (poly_regression.py:118).
        Returns ``(moments, fit_mask, x_limits, y_limits)``; the limits ([K, G, 2] f64 (lo, hi), None without a
        stretch) belong to THIS call's data — nothing is kept on the instance, so one synthesizer can serve
        several streams / threads.  With a stretch: mask first, then the limits, then the moments; ``reduce``
        (a global fit with stretch_scope="fit") sums the percentile histograms across processes, so the limits are
        those of every process's masked pixels."""
        xl = yl = None
        if self.stretch is not None:
            fit_mask = self.stretch_mask(bands, s2_ref, valid, fit_mask, groups=groups)
            xl, yl = self.stretch_limits([(bands, s2_ref, fit_mask)], reduce, groups=groups)
        mom, fm = self._fit_moments(bands, s2_ref, valid, fit_mask, xl, yl, groups=groups, exchange=exchange)
        return mom, fm, xl, yl

    def _fit_moments(self, bands, s2_ref, valid, fit_mask, xl, yl, *, groups=1, exchange=None):
        """``(moments, fit_mask)``: with ``y_finite`` and no stretch the moment kernel builds the mask from ``valid``
        (no separate mask launch); otherwise ``fit_mask`` is the mask, with the stretch limits ``xl`` / ``yl`` if any."""
        if self.y_finite and self.stretch is None:
            return kernels.fit_moments(bands, s2_ref, valid, self.deg, groups=groups, gate_k=self.gate_k, gate_gt=0.0,
                                       y_finite=True, exchange=exchange)
        return kernels.fit_moments(bands, s2_ref, fit_mask, self.deg, groups=groups, mask_given=True, x_stretch=xl,
                                   y_stretch=yl, exchange=exchange)

    def stretch_mask(self, bands, s2_ref, valid, fit_mask, *, groups=1):
        """The pixels the stretch percentiles and the fit are taken over (with ``y_finite``: rebuilt so that
        non-finite reference pixels drop out, poly_regression.py:118)."""
        if self.y_finite:
            return kernels.fit_mask(bands, valid, gate_k=self.gate_k, gate_gt=0.0, y=s2_ref, groups=groups)
        return fit_mask

    def stretch_limits(self, units, reduce=None, *, groups=1):
        """``(x_limits, y_limits)`` over the union of ``units`` ([(bands, s2_ref, mask), ...]) and, when ``reduce`` is
        given, of every process's units.  One unit on one process takes the one-pass select
        (``kernels.masked_percentiles``, same bits, faster); anything more the union select."""
        if reduce is None and len(units) == 1:
            bands, s2_ref, mask = units[0]
            return kernels.masked_percentiles(bands, mask, self.stretch, groups=groups, y=s2_ref)
        return kernels.masked_percentiles_union(units, self.stretch, reduce=reduce or _no_reduce, K=self.K, pair=True,
                                                device=self.device)

    def _check_global(self, exchange, allreduce) -> bool:
        """Whether a call's fit is global across ranks (``exchange=`` / ``allreduce=True`` with more than one
        process); raises for a stretch whose limits would be per granule, and for ``exchange=`` with OT targets."""
        self._no_ot_exchange(exchange)
        global_fit = (exchange is not None and exchange.world > 1) or (allreduce and hdist.world()[1] > 1)
        if global_fit:
            self._no_global_stretch("exchange= / allreduce=True")
        return global_fit

    def _no_ot_exchange(self, exchange) -> None:
        """The peer exchange carries moment sums; an OT fit forms no per-rank moments that could be summed."""
        if exchange is not None and self.targets == "ot":
            raise ValueError("exchange= cannot carry an OT fit (targets=\"ot\"): the peer exchange sums moments, and the "
                             "OT targets are drawn over the union of every rank's rows; use allreduce=True / group=")

    def _global_reduce(self, group):
        """The SUM all-reduce of the percentile histograms of a global fit (None for one process)."""
        if self.stretch is None or hdist.group_size(group) == 1:
            return None
        return lambda t: hdist.allreduce_moments(t, group)

    def _no_global_stretch(self, what: str) -> None:
        """With stretch_scope="granule" the percentile limits are per granule (color.py:30-32 sees one image): moments
        of differently normalised granules must not be summed into one polynomial."""
        if self.stretch is not None and self.stretch_scope == "granule":
            raise ValueError(f"stretch=(pmin, pmax) cannot be combined with a global fit ({what}): every granule would be "
                             "normalised by its own percentiles before the moments are summed; pass "
                             "stretch_scope=\"fit\" for limits over the whole fit, fit per granule, or stretch with "
                             "limits of your own before calling")

    @property
    def _clip_bounds(self) -> tuple:
        """``(lo, hi)`` of the apply's clip; lo > hi (``clip=None``) clips nothing."""
        return self.clip if self.clip is not None else (1.0, 0.0)

    # ------------------------------------------------------------------ the fit and apply of every entry point
    def _fit_apply(self, units: Iterable[_Unit], *, groups: int = 1, global_fit: bool = False, group=None,
                   exchange=None, allreduce: bool = False, summed: bool = False) -> List[PairResult]:
        """Fit and solve / apply ``units`` (this rank's images of one fit, in order) -> one PairResult per unit.

        With a stretch or OT targets each unit's fit mask is taken as the unit arrives (:meth:`stretch_mask`).  The
        stretch limits cover every unit and, with ``global_fit``, every rank of ``group``.  The moments are the one
        unit's (``groups`` series per plane for a tile batch), the fixed-order sum of the units' with ``summed``, or
        :meth:`_ot_moments` (over every rank of ``group`` with ``allreduce``).  Paired moments are made global by
        ``exchange`` (a ``dist.PeerExchange``: the moment kernel, or with ``summed`` the sum, publishes; the first
        solve / apply consumes and returns the global sums for the other units; a rank with no unit still consumes)
        or else, with ``allreduce``, by one all-reduce over ``group``."""
        if self.stretch is not None or self.targets == "ot":
            units = (replace(u, fit_mask=self.stretch_mask(u.bands, u.s2_ref, u.valid, u.fit_mask, groups=groups))
                     for u in units)
        units = list(units)
        ex = exchange.next() if exchange is not None and exchange.world > 1 else None
        xl = yl = None
        if self.stretch is not None:
            reduce = self._global_reduce(group) if global_fit else None
            xl, yl = self.stretch_limits([(u.bands, u.s2_ref, u.fit_mask) for u in units], reduce, groups=groups)
        min_count, info = self.min_count, None
        with torch.cuda.device(self.device):
            if self.targets == "ot":
                mom, min_count, info = self._ot_moments([(u.bands, u.s2_ref, u.fit_mask) for u in units], xl, yl,
                                                        group, allreduce)
            else:
                moms = []
                for u in units:
                    m, u.fit_mask = self._fit_moments(u.bands, u.s2_ref, u.valid, u.fit_mask, xl, yl, groups=groups,
                                                      exchange=None if summed else ex)
                    moms.append(m)
                if summed:
                    like = torch.empty((self.K, 3 * self.deg + 2), dtype=torch.float64, device=self.device)
                    mom = kernels.moments_sum([m.view(self.K, -1) for m in moms], like=like, exchange=ex)
                else:
                    (mom,) = moms
                if allreduce and ex is None:
                    hdist.allreduce_moments(mom, group)
            lo, hi = self._clip_bounds
            if ex is not None and not units:
                # nothing to apply here, but the exchange must be consumed (the slot parity protocol lets a rank run at
                # most one epoch ahead of its own consumption)
                x0 = torch.zeros((self.K, 1), dtype=torch.float32, device=self.device)
                m0 = torch.zeros(1, dtype=torch.uint8, device=self.device)
                kernels.poly_solve_apply(x0, mom, m0, self.deg, min_count=min_count, lo=lo, hi=hi, exchange=ex)
            out = []
            for u in units:
                gmom = torch.empty_like(mom) if ex is not None else None
                coeffs, matched = kernels.poly_solve_apply(u.bands, mom, u.fit_mask, self.deg, groups=groups,
                                                           min_count=min_count, lo=lo, hi=hi, out=u.matched_out,
                                                           x_stretch=xl, exchange=ex, moments_out=gmom)
                if gmom is not None:          # the global sums: the later units solve them without the exchange
                    mom, ex = gmom, None
                lead = u.bands.shape[1:-2]    # (T,) for a tile batch
                out.append(PairResult(u.bands, matched, coeffs.view(self.K, *lead, self.deg + 1), u.valid,
                                      u.fit_mask.view(u.valid.shape), u.diag, mom.view(self.K, *lead, -1), u.ortho,
                                      self.band_names, xl, yl, grid=u.grid, ot_info=info))
        return out

    # ------------------------------------------------------------------ one granule
    def synthesize(self, raw: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor, s2_ref: torch.Tensor, *,
                   transpose_raw_yx: bool = False, materialize_ortho: bool = False, group=None,
                   allreduce: bool = False, bands_out=None, matched_out=None, exchange=None,
                   raw_row0: int = 0, raw_rows_total: Optional[int] = None) -> PairResult:
        """raw [Hr, Wr, B] f32, GLT planes [Ho, Wo] int32, s2_ref [K, Ho, Wo] f32 — all CUDA tensors.
        Three launches (+ the moment finalize): glt_srf, fit_moments, poly_solve_apply.
        Global fit across ranks: ``exchange`` (a ``dist.PeerExchange``: moments travel over NVLink peer memory
        inside the finalize / solve kernels) or ``allreduce=True`` (one NCCL all-reduce between the two)."""
        global_fit = self._check_global(exchange, allreduce)
        unit = self._planes(raw, glt_x, glt_y, s2_ref, transpose_raw_yx, materialize_ortho=materialize_ortho,
                            bands_out=bands_out, raw_row0=raw_row0, raw_rows_total=raw_rows_total)
        unit.matched_out = matched_out
        return self._fit_apply([unit], global_fit=global_fit, group=group, exchange=exchange, allreduce=allreduce)[0]

    def _planes(self, raw, glt_x, glt_y, s2_ref, transpose_raw_yx=False, **kw) -> _Unit:
        """glt_srf with the fit mask, on the ortho grid."""
        fm = torch.empty(glt_x.shape, dtype=torch.bool, device=raw.device)
        bands, valid, diag, ortho = self.bands_from_raw(raw, glt_x, glt_y, transpose_raw_yx=transpose_raw_yx,
                                                        fit_mask_out=fm, **kw)
        return _Unit(bands, s2_ref, valid, fm, diag, ortho)

    # ------------------------------------------------------------------ one granule on the Sentinel-2 grid
    def synthesize_on_s2_grid(self, raw: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor, s2_ref: torch.Tensor,
                              target: S2Target, *, transpose_raw_yx: bool = False, bands_out=None,
                              matched_out=None, group=None, allreduce: bool = False, exchange=None) -> PairResult:
        """The pair on the Sentinel-2 UTM grid ``target`` (:func:`hsr_b200.EMIT_data.warp.s2_target`), where the
        reference fits: ``s2_ref`` [K, Hd, Wd] f32 is the S2 stack on that grid.  Instead of warping the B-band ortho
        cube and integrating the SRF over it (nc_to_envi's gdalwarp, then synth.py:9-45), the K pseudo-S2 planes of
        the fused GLT + SRF pass are warped (``kernels.warp_planes``, GLT-valid pixels only): both steps are linear and
        the warp's tap weights are the same for every band, so the result is the same up to fp rounding.
        Stages: glt_srf, the target's cached coordinates, warp_planes, then the fit and solve / apply of
        :meth:`synthesize` (stretch, ``y_finite``, gate band and clip as there, on the S2-grid planes).
        ``bands``, ``matched``, ``valid`` and ``fit_mask`` of the result are on the target grid, ``diag`` is the GLT
        diagnostics of the source pass and ``grid`` is ``target``.  ``group`` / ``allreduce`` / ``exchange``: a global
        fit across ranks, one granule per rank, as in :meth:`synthesize` (with ``stretch_scope="fit"`` the limits are
        those of every rank's pixels).  Deviation from the reference: a GLT-valid raw spectrum holding the nodata value
        in some or all of its bands is used as data (DESIGN section 7)."""
        self._check_s2_ref(s2_ref, target.shape)
        global_fit = self._check_global(exchange, allreduce)
        unit = self._planes_on_grid(raw, glt_x, glt_y, s2_ref, target, transpose_raw_yx, bands_out)
        unit.matched_out = matched_out
        return self._fit_apply([unit], global_fit=global_fit, group=group, exchange=exchange, allreduce=allreduce)[0]

    def _check_s2_ref(self, s2_ref, shape) -> None:
        Hd, Wd = shape
        if tuple(s2_ref.shape) != (self.K, Hd, Wd):
            raise ValueError(f"s2_ref must be [K={self.K}, {Hd}, {Wd}] on the target grid, got {tuple(s2_ref.shape)}")

    def _planes_on_grid(self, raw, glt_x, glt_y, s2_ref, target: S2Target, transpose_raw_yx=False,
                        bands_out=None) -> _Unit:
        """glt_srf, then the plane warp onto ``target``."""
        src, valid, diag, _ = self.bands_from_raw(raw, glt_x, glt_y, transpose_raw_yx=transpose_raw_yx)
        fm = torch.empty(target.shape, dtype=torch.bool, device=src.device)
        bands, dvalid, fm = kernels.warp_planes(src, valid, target.coords(src.device), target.scales,
                                                kernel=target.kernel, fill_out=self.fill_out, gate_k=self.gate_k,
                                                gate_gt=0.0, out=bands_out, fit_mask_out=fm)
        return _Unit(bands, s2_ref, dvalid, fm, diag, grid=target)

    # ------------------------------------------------------------------ a row slab of a mosaic
    def synthesize_slab(self, raw, glt_x: torch.Tensor, glt_y: torch.Tensor, s2_ref: torch.Tensor, *,
                        transpose_raw_yx: bool = False, stage: Optional[torch.Tensor] = None, **kw) -> PairResult:
        """One row slab of a large ortho grid (BASELINE configs[4]; ``dist.shard_rows``) with PER-SLAB RAW STAGING
        (SURVEY 7.3-6): the slab's GLT references a band of the raw mosaic, so only the raw rows between the smallest
        and the largest ``gy`` of the slab are brought to the device.

        raw: the whole raw mosaic [Hr, Wr, B] f32 — a (pinned) HOST tensor / numpy array, or a CUDA tensor (then the
        window is just a view); glt_x / glt_y: the slab's rows of the GLT (CUDA int32); s2_ref: the slab's rows of the
        reference planes.  ``stage``: optional preallocated CUDA buffer the window is copied into (flat f32, at least
        rows * Wr * B elements).  Other keywords as :meth:`synthesize` (``exchange=`` / ``allreduce=`` make the fit
        global over the slabs).  The result's ``raw_rows`` holds the staged [row0, row1) range."""
        with torch.cuda.device(self.device):
            win, lo, hi, d0 = self._stage_raw(raw, glt_x, glt_y, transpose_raw_yx, stage)
            res = self.synthesize(win, glt_x, glt_y, s2_ref, transpose_raw_yx=transpose_raw_yx, raw_row0=lo,
                                  raw_rows_total=d0, **kw)
            return _slab_checked(res, (lo, hi))

    def _stage_raw(self, raw, glt_x, glt_y, transpose_raw_yx, stage):
        """(window on the device, lo, hi, raw rows): the raw rows [lo, hi) of ``raw`` (a numpy array or a host / CUDA
        tensor of ``raw rows`` rows) that the GLT rows reference, copied into ``stage`` (or a new device buffer) when
        ``raw`` is in host memory."""
        raw = _as_tensor(raw)
        d0, d1 = int(raw.shape[0]), int(raw.shape[1])
        Hr, Wr = (d1, d0) if transpose_raw_yx else (d0, d1)
        lo, hi = kernels.glt_row_range(glt_x, glt_y, Hr, Wr, transpose_raw_yx=transpose_raw_yx).tolist()
        if hi == 0:                       # no valid entry in this slab: any one row will do
            lo, hi = 0, 1
        win = raw[lo:hi]
        if not win.is_cuda:
            n = win.numel()
            buf = stage if stage is not None else torch.empty(n, dtype=torch.float32, device=self.device)
            if buf.numel() < n:
                raise ValueError(f"stage holds {buf.numel()} floats, the slab's raw window needs {n}")
            dst = buf.view(-1)[:n].view(win.shape)
            dst.copy_(win, non_blocking=win.is_pinned())
            win = dst
        return win, lo, hi, d0

    # ------------------------------------------------------------------ a row band of a mosaic on the Sentinel-2 grid
    def synthesize_slab_on_s2_grid(self, raw, glt_x: torch.Tensor, glt_y: torch.Tensor, s2_ref: torch.Tensor,
                                   target: S2Target, rows, *, transpose_raw_yx: bool = False,
                                   stage: Optional[torch.Tensor] = None, group=None, allreduce: bool = False,
                                   exchange=None) -> PairResult:
        """One band ``rows`` = (t0, t1) of the target rows of a mosaic on the Sentinel-2 grid ``target``
        (``dist.shard_rows(target.shape[0], ...)`` deals the bands), staging only what the band reads: the
        coordinates of its rows, the ortho rows [o0, o1) its filter reaches (``kernels.warp_src_row_range``), the raw
        rows the GLT rows [o0, o1) reference (``kernels.glt_row_range``), then glt_srf on those GLT rows through a raw
        view, the plane warp over the ortho window and the fit / solve / apply of :meth:`synthesize_on_s2_grid`.

        raw: the whole raw mosaic [Hr, Wr, B] f32 — a (pinned) host tensor / numpy array or a CUDA tensor; glt_x /
        glt_y: the whole GLT [Ho, Wo] on the device; s2_ref: [K, t1 - t0, Wd], the band's rows of the reference.
        ``stage``: as in :meth:`synthesize_slab`.  ``group`` / ``allreduce`` / ``exchange``: a global fit over the bands
        of every rank (with ``stretch_scope="fit"``, limits over every band).  Stitched along rows, the bands' planes
        and masks are bit-identical to one :meth:`synthesize_on_s2_grid` call: the windowed warp reads the same source
        values with the same weights.  A band that reads no source row (no pixel centre inside the ortho grid) stages
        nothing and yields fill, and still takes part in the exchange / all-reduce / percentile reduce.

        The result's ``raw_rows`` and ``ortho_rows`` hold the staged [row0, row1) ranges.  ``diag`` is the GLT
        diagnostics of the staged ortho rows; neighbouring bands overlap by the filter footprint, so the bands' diag
        do NOT sum to the granule's.  Raises ``RuntimeError`` when a GLT entry or a filter tap fell outside the staged
        rows (after the fit, so that no rank is left waiting in the exchange)."""
        Hd, Wd = target.shape
        t0, t1 = int(rows[0]), int(rows[1])
        if not 0 <= t0 < t1 <= Hd:
            raise ValueError(f"rows must satisfy 0 <= t0 < t1 <= {Hd}, got {tuple(rows)}")
        self._check_s2_ref(s2_ref, (t1 - t0, Wd))
        global_fit = self._check_global(exchange, allreduce)
        Ho, Wo = glt_x.shape
        with torch.cuda.device(self.device):
            coords = target.coords(self.device, rows=(t0, t1))
            o0, o1 = kernels.warp_src_row_range(coords, (Ho, Wo), target.scales, kernel=target.kernel).tolist()
            if o1 == 0:                       # no pixel centre inside the ortho grid: nothing to stage
                o0 = o1 = lo = hi = 0
                src = torch.empty((self.K, 0, Wo), dtype=torch.float32, device=self.device)
                valid = torch.empty((0, Wo), dtype=torch.bool, device=self.device)
                diag = torch.zeros(4, dtype=torch.int64, device=self.device)
            else:
                gx, gy = glt_x[o0:o1], glt_y[o0:o1]
                win, lo, hi, d0 = self._stage_raw(raw, gx, gy, transpose_raw_yx, stage)
                src, valid, diag, _ = self.bands_from_raw(win, gx, gy, transpose_raw_yx=transpose_raw_yx, raw_row0=lo,
                                                          raw_rows_total=d0)
            outside = torch.zeros(1, dtype=torch.int64, device=self.device)
            fm = torch.empty((t1 - t0, Wd), dtype=torch.bool, device=self.device)
            bands, dvalid, fm = kernels.warp_planes(src, valid, coords, target.scales, kernel=target.kernel,
                                                    fill_out=self.fill_out, gate_k=self.gate_k, gate_gt=0.0,
                                                    fit_mask_out=fm, src_row0=o0, src_rows_total=Ho, outside=outside)
            res = self._fit_apply([_Unit(bands, s2_ref, dvalid, fm, diag, grid=target)], global_fit=global_fit,
                                  group=group, exchange=exchange, allreduce=allreduce)[0]
            return _slab_checked(res, (lo, hi), (o0, o1), outside)

    # ------------------------------------------------------------------ a batch of equal tiles
    def synthesize_tiles(self, raw_tiles: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor,
                         s2_ref: torch.Tensor) -> PairResult:
        """Tile batch (tiles_helpers shape contract): raw_tiles [T, h, w, B], GLT planes [T, h, w] with
        per-tile 1-based indices, s2_ref [K, T, h, w].  One launch per stage; T*K independent fits.
        The tiles are stacked along rows; the kernel itself offsets tile t's GLT rows by t*h and keeps an entry that
        points past its own tile out of bounds (hsr_raw_view_t.batch_*), so the GLT is used as delivered."""
        if self.targets == "ot":
            raise ValueError("synthesize_tiles fits T * K independent pixel-paired series; OT targets (targets=\"ot\") "
                             "are not available for tile batches")
        T, h, w, B = raw_tiles.shape
        u = self._planes(raw_tiles.reshape(T * h, w, B), glt_x.reshape(T * h, w), glt_y.reshape(T * h, w), s2_ref,
                         tile_rows=(h, h))
        u = replace(u, bands=u.bands.view(self.K, T, h, w), valid=u.valid.view(T, h, w),
                    fit_mask=u.fit_mask.view(T, h, w), diag=u.diag[:3])
        return self._fit_apply([u], groups=T)[0]

    # ------------------------------------------------------------------ many granules, one global fit
    def synthesize_sharded(self, granules: Sequence[dict], *, group=None, exchange=None) -> List[PairResult]:
        """Granules owned by THIS rank (dicts with raw, glt_x, glt_y, s2_ref, optionally "target": an ``S2Target``, for
        a granule synthesised on that Sentinel-2 grid as :meth:`synthesize_on_s2_grid` does, s2_ref then being on the
        target grid and the result's ``grid`` the target) — BASELINE configs[3]; the fit is
        GLOBAL: the local moments are summed in a fixed order (``kernels.moments_sum``), summed across ranks once —
        over NVLink peer memory when ``exchange`` (a ``dist.PeerExchange``) is given, else one all-reduce (NCCL /
        gloo) — and solved redundantly.  A rank that was dealt no granule still takes part in the exchange.
        With ``stretch_scope="fit"`` the stretch limits are the percentiles of every granule on every rank (their
        histograms are summed over ``group`` with ``dist.all_reduce`` also when the moments go through ``exchange``).
        With ``targets="ot"`` the fit is the OT fit over every granule's rows on every rank (``exchange`` raises)."""
        self._no_global_stretch("synthesize_sharded")
        self._no_ot_exchange(exchange)

        def unit(g):
            target, tr = g.get("target"), g.get("transpose_raw_yx", False)
            if target is None:
                return self._planes(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"], tr)
            self._check_s2_ref(g["s2_ref"], target.shape)
            return self._planes_on_grid(g["raw"], g["glt_x"], g["glt_y"], g["s2_ref"], target, tr)
        # a generator: each granule's fit mask is taken right after its planes
        return self._fit_apply((unit(g) for g in granules), global_fit=True, group=group, exchange=exchange,
                               allreduce=True, summed=True)

    # ------------------------------------------------------------------ OT targets
    def _ot_moments(self, units, xl, yl, group, union):
        """``fit_ot_poly_rgb`` over the concatenation, in (rank, unit) order, of the rows of ``units`` ([(bands,
        s2_ref, mask)]) of this process or, with ``union``, of every rank of ``group``.  Returns ``(moments [K,
        3*deg+2], min_count, ot_info)`` for ``poly_solve_apply``: the moments of (X, Ybar) with min_count 0, or zeros
        with min_count 1 (the identity) when the union has fewer than ``min_count`` X or Y rows.

        Each unit's rows are compacted on the device; the per-unit counts come to the host and the per-rank totals are
        summed with one all-reduce ([world, 2], each rank filling its own row), so every rank knows where every rank's
        rows start in the union and draws the same samples.  Each rank gathers the samples it owns into [ns, K] / [nt, K]
        buffers prefilled with -0.0 and one SUM all-reduce assembles them: -0.0 + v == v for every v, so each row
        arrives with its owner's bits whatever the reduction order."""
        K, dev = self.K, self.device
        world = hdist.group_size(group) if union else 1
        rank = torch.distributed.get_rank(group) if world > 1 else 0
        lists = [kernels.compact_planes_pair(b, y, m, x_stretch=xl, y_stretch=yl) for b, y, m in units]
        cnt = torch.stack([torch.cat([cx, cy]) for _, cx, _, cy in lists]) if lists else \
            torch.zeros((0, 2), dtype=torch.int64, device=dev)
        tot = torch.zeros((world, 2), dtype=torch.float64, device=dev)
        tot[rank] = cnt.sum(0).to(torch.float64)
        if world > 1:
            hdist.allreduce_moments(tot, group)
        cnt_h = cnt.tolist()
        tot_h = [[int(v) for v in row] for row in tot.tolist()]
        nx, ny = sum(r[0] for r in tot_h), sum(r[1] for r in tot_h)
        M = 3 * self.deg + 2
        if nx < self.min_count or ny < self.min_count:                    # poly_regression.py:38-41
            return torch.zeros((K, M), dtype=torch.float64, device=dev), 1, None
        rng = np.random.default_rng(self.seed)                            # :31
        ns, nt = min(self.n_samples, nx), min(self.n_samples, ny)
        sel = (rng.choice(nx, size=ns, replace=False).astype(np.int64),   # :46-47
               rng.choice(ny, size=nt, replace=False).astype(np.int64))
        buf = torch.full(((ns + nt) * K,), -0.0, dtype=torch.float64, device=dev)
        XY = (buf[:ns * K].view(ns, K), buf[ns * K:].view(nt, K))
        for side in (0, 1):                                               # X from the bands, Y from the reference
            owned = ot_owned_rows(sel[side], [r[side] for r in tot_h], rank, [c[side] for c in cnt_h])
            for (bands, s2_ref, _), lst, (rows, local) in zip(units, lists, owned):
                if rows.size:
                    kernels.gather_planes_f64((bands, s2_ref)[side], lst[2 * side], torch.from_numpy(local).to(dev),
                                              stretch=(xl, yl)[side], dst=torch.from_numpy(rows).to(dev), out=XY[side])
        if world > 1:
            hdist.allreduce_moments(buf, group)
        if not units:                                                     # nothing to apply on this rank
            return torch.zeros((K, M), dtype=torch.float64, device=dev), 1, None
        ybar, info = kernels.sinkhorn_barycentric(XY[0], XY[1], self.reg, self.numItermax, self.stopThr)   # :49-56
        mom = kernels.polyfit_moments_f64(XY[0], ybar, self.deg)                                            # :58-60
        return mom, 0, tuple(info.tolist())

    # ------------------------------------------------------------------ the step to the finer (S2 10 m) resolution
    def matched_fine(self, results, factor: int = 6, *, group=None, out=None):
        """Colour-matched planes on the ``factor``-times finer aligned grid — the reference script's last step
        (s2_emit/poly_regression.py:150-162), for the K planes of a pair result: ``x10 = bilinear x factor`` of the
        result's (unstretched) ``bands``, ``mask10 = isfinite(x10).all(0)``, with ``stretch`` the percentiles of x10
        under mask10 (``lim10``) and ``xs = clip((x10 - lo) / (hi - lo + 1e-12), 0, 1)`` on every pixel (else
        ``xs = x10``), ``(f32) polyval(coeffs[k], xs)`` where mask10, then every pixel clipped to ``clip``.  On an S2
        target grid (snapped to the S2 origin at an integer ratio) factor 6 gives the S2 10 m grid.  Fill pixels
        (``fill_out``) are finite and therefore data here, as in the reference (DESIGN section 7).

        ``results``: one ``PairResult`` -> one ``FineResult``; a sequence of the results of ONE global fit (e.g.
        ``synthesize_sharded``, possibly empty on a rank that holds no granule) -> a list.  The 10 m limits follow the
        60 m ones: one result has its own; several (``stretch_scope="fit"``) share the union over all of them and, with
        ``group``, over every rank of the group — every rank must then call, also with no result.  The fine planes are
        never materialised: a fine mask, a union select over fine values formed from the 60 m planes in each of its
        four passes, and one fused apply (``kernels.bilinear_fine_mask``, ``kernels.masked_percentiles_union(factor=)``,
        ``kernels.bilinear_apply``).  ``out``: a [K, f*H, f*W] f32 tensor (one result) or a list of them.
        Raises ``ValueError`` for tile batches, row slabs (the upsample at a slab edge needs the neighbouring slab's
        rows) and ``factor < 1``."""
        single = isinstance(results, PairResult)
        rs = [results] if single else list(results)
        f = int(factor)
        if f < 1 or f != factor:
            raise ValueError(f"factor must be an integer >= 1, got {factor!r}")
        for r in rs:
            if r.coeffs.dim() != 2 or r.bands.dim() != 3:
                raise ValueError("matched_fine takes granule results: tile batches (coeffs [K, T, deg+1]) are not covered")
            if r.raw_rows is not None or r.ortho_rows is not None:
                raise ValueError("matched_fine does not take row slabs: the upsample at a slab edge needs the "
                                 "neighbouring slab's rows")
        outs = [out] if single else (list(out) if out is not None else [None] * len(rs))
        if len(outs) != len(rs):
            raise ValueError(f"out holds {len(outs)} tensors for {len(rs)} results")
        with torch.cuda.device(self.device):
            # the select needs mask10 before the apply; without a stretch the apply writes it
            masks = [kernels.bilinear_fine_mask(r.bands, f) if self.stretch is not None else
                     torch.empty((r.bands.shape[1] * f, r.bands.shape[2] * f), dtype=torch.bool, device=self.device)
                     for r in rs]
            xl = None
            if self.stretch is not None:
                world = hdist.group_size(group) if group is not None else 1
                if len(rs) > 1 or world > 1:
                    self._no_global_stretch("matched_fine over several results / ranks")
                reduce = self._global_reduce(group) if group is not None else None
                xl = kernels.masked_percentiles_union([(r.bands, m) for r, m in zip(rs, masks)], self.stretch,
                                                      reduce=reduce or _no_reduce, K=self.K, pair=False,
                                                      device=self.device, factor=f)
            lo, hi = self._clip_bounds
            fine = []
            for r, m, o in zip(rs, masks, outs):
                matched, _ = kernels.bilinear_apply(r.bands, f, r.coeffs, x_stretch=xl, lo=lo, hi=hi, out=o, mask_out=m)
                win = None
                if r.grid is not None:
                    win = (int(r.grid.s2_window[0]) * f, int(r.grid.s2_window[1]) * f)
                fine.append(FineResult(matched, m, xl, f, win))
        return fine[0] if single else fine


def ot_owned_rows(sel, rank_counts, rank: int, unit_counts):
    """The samples of a union draw that one rank's units own.  ``sel``: indices into the concatenation of every rank's
    rows in (rank, unit) order; ``rank_counts``: rows per rank; ``unit_counts``: rows per unit of ``rank``.  Returns one
    ``(rows, local)`` pair per unit: the positions r in ``sel`` whose row lies in that unit, and the row's index within
    the unit (``sel[rows] - unit offset``), both int64."""
    sel = np.asarray(sel, dtype=np.int64)
    off = int(sum(rank_counts[:rank]))
    out = []
    for c in unit_counts:
        rows = np.flatnonzero((sel >= off) & (sel < off + int(c))).astype(np.int64)
        out.append((rows, sel[rows] - off))
        off += int(c)
    return out


def _as_tensor(raw):
    """A numpy raw mosaic as a (host) tensor; tensors pass through."""
    return torch.from_numpy(raw) if isinstance(raw, np.ndarray) else raw


def _slab_checked(res: PairResult, raw_rows: tuple, ortho_rows: Optional[tuple] = None,
                  outside: Optional[torch.Tensor] = None) -> PairResult:
    """A row slab's result: raises ``RuntimeError`` when a valid GLT entry (``diag[3]``) or, on the S2 grid, a filter
    tap (``outside``) fell outside the staged rows — only now, after the fit and apply, so that no rank is left waiting
    in the exchange — then keeps the three GLT diagnostics and records the staged ranges."""
    raw_missed, *tap_missed = torch.cat([res.diag[3:]] + ([outside] if outside is not None else [])).tolist()
    if raw_missed:
        raise RuntimeError(f"{raw_missed} valid GLT entries fell outside the staged raw rows [{raw_rows[0]}, {raw_rows[1]})")
    if tap_missed and tap_missed[0]:
        raise RuntimeError(f"{tap_missed[0]} target pixels needed ortho rows outside the staged rows "
                           f"[{ortho_rows[0]}, {ortho_rows[1]})")
    res.diag, res.raw_rows, res.ortho_rows = res.diag[:3], raw_rows, ortho_rows
    return res


class HostGranuleStream:
    """Granules that live in HOST memory, streamed through one GPU: upload, pair synthesis and download of
    consecutive granules overlap on three CUDA streams (H2D / compute / D2H) over ``depth`` device slots.

    This is the end-to-end entry point for callers that hold numpy / pinned host buffers (the reference's
    callers do: it reads an ENVI file into host memory, ``s2_emit/emit_io.py:7-16``).  PCIe is the bound
    (1.97 GB up, 0.14 GB down per granule); the kernels (0.5 ms) and the download of granule i hide behind
    the upload of granule i + 1.

        stream = HostGranuleStream(ps, raw_shape=(Hr, Wr, B), ortho_shape=(Ho, Wo))
        for g in granules:
            stream.submit(g.raw, g.glt_x, g.glt_y, g.s2_ref, out=host_result)   # asynchronous
        stream.drain()
    """

    def __init__(self, ps: PairSynthesizer, raw_shape, ortho_shape, *, depth: int = 2, allreduce: bool = False,
                 exchange=None):
        if ps.targets == "ot":
            raise ValueError("HostGranuleStream overlaps upload, compute and download on three streams; an OT fit "
                             "(targets=\"ot\") needs a host round trip per granule for the sample draw, so nothing "
                             "would overlap: call synthesize per granule instead")
        self.ps, self.depth, self.allreduce, self.exchange = ps, int(depth), bool(allreduce), exchange
        dev = ps.device
        Hr, Wr, B = raw_shape
        Ho, Wo = ortho_shape
        self.n_o = Ho * Wo
        self.h2d, self.comp, self.d2h = (torch.cuda.Stream(dev) for _ in range(3))
        self.slots = []
        for _ in range(self.depth):
            s2 = kernels.alloc_planes(ps.K, (Ho, Wo), dev)
            self.slots.append({
                "raw": torch.empty((Hr, Wr, B), dtype=torch.float32, device=dev),
                "gx": torch.empty((Ho, Wo), dtype=torch.int32, device=dev),
                "gy": torch.empty((Ho, Wo), dtype=torch.int32, device=dev),
                "s2": s2, "bands": kernels.alloc_planes(ps.K, (Ho, Wo), dev),
                "matched": kernels.alloc_planes(ps.K, (Ho, Wo), dev),
                "uploaded": torch.cuda.Event(), "computed": torch.cuda.Event(), "downloaded": torch.cuda.Event(),
                "res": None,
            })
        self.stride = self.slots[0]["s2"].stride(0)       # padded plane stride (floats)
        self.i = 0

    def host_buffers(self):
        """Pinned host buffers shaped for one granule's results: planes keep the padded device stride so that
        every transfer is one contiguous copy."""
        K = self.ps.K
        Ho, Wo = self.slots[0]["gx"].shape
        return {"matched": torch.empty((K, self.stride), dtype=torch.float32, pin_memory=True),
                "valid": torch.empty((Ho, Wo), dtype=torch.bool, pin_memory=True),
                "coeffs": torch.empty((K, self.ps.deg + 1), dtype=torch.float64, pin_memory=True)}

    @staticmethod
    def _flat(planes: torch.Tensor, stride: int) -> torch.Tensor:
        """The [K, stride] buffer behind padded planes."""
        return torch.as_strided(planes, (planes.shape[0], stride), (stride, 1))

    def submit(self, h_raw, h_gx, h_gy, h_s2, out) -> None:
        """h_raw [Hr, Wr, B] f32, h_gx / h_gy [Ho, Wo] int32, h_s2 [K, stride] (padded) or [K, Ho, Wo] f32 — pinned
        host tensors; ``out``: dict from :meth:`host_buffers`.  Returns immediately."""
        sl = self.slots[self.i % self.depth]
        self.i += 1
        self.h2d.wait_event(sl["downloaded"])             # the slot's previous results have left the device
        with torch.cuda.stream(self.h2d):
            sl["raw"].copy_(h_raw, non_blocking=True)
            sl["gx"].copy_(h_gx, non_blocking=True)
            sl["gy"].copy_(h_gy, non_blocking=True)
            if h_s2.dim() == 2 and h_s2.shape[1] == self.stride:
                self._flat(sl["s2"], self.stride).copy_(h_s2, non_blocking=True)
            else:
                sl["s2"].copy_(h_s2, non_blocking=True)
            sl["uploaded"].record(self.h2d)
        self.comp.wait_event(sl["uploaded"])
        with torch.cuda.stream(self.comp):
            res = self.ps.synthesize(sl["raw"], sl["gx"], sl["gy"], sl["s2"], allreduce=self.allreduce,
                                     bands_out=sl["bands"], matched_out=sl["matched"], exchange=self.exchange)
            sl["computed"].record(self.comp)
        sl["res"] = res
        self.d2h.wait_event(sl["computed"])
        with torch.cuda.stream(self.d2h):
            for t in (res.valid, res.coeffs):
                t.record_stream(self.d2h)
            if out["matched"].dim() == 2 and out["matched"].shape[1] == self.stride:
                out["matched"].copy_(self._flat(sl["matched"], self.stride), non_blocking=True)
            else:
                out["matched"].copy_(sl["matched"], non_blocking=True)
            out["valid"].copy_(res.valid, non_blocking=True)
            out["coeffs"].copy_(res.coeffs, non_blocking=True)
            sl["downloaded"].record(self.d2h)

    def drain(self) -> None:
        """Make the CURRENT stream wait for everything submitted so far (results are in the host buffers once
        the current stream has been synchronised)."""
        cur = torch.cuda.current_stream(self.ps.device)
        for sl in self.slots:
            cur.wait_event(sl["downloaded"])
