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
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import torch

from . import dist as hdist
from . import kernels
from ._host import cuda_device, to_device
from .s2_emit.srf import srf_fold_weights

NO_DATA_VALUE = kernels.NO_DATA_VALUE
STRETCH_SCOPES = ("granule", "fit")


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


class PairSynthesizer:
    """Holds the folded SRF weights on the device and runs the fused pass for granules or tile batches."""

    def __init__(self, emit_w, srf_dict: Dict[str, tuple], good_mask=None, *, deg: int = 2,
                 fill: float = NO_DATA_VALUE, min_count: int = 200, gate_band: Optional[str] = None,
                 clip=(0.0, 1.0), y_finite: bool = False, stretch=None, stretch_scope: str = "granule", device=None):
        """``stretch=(pmin, pmax)`` inserts the shared percentile stretch of s2_emit/color.py:25-34 between the
        SRF synthesis and the fit, as the reference's script does (poly_regression.py:126-127): both images are
        stretched with their own masked percentiles, the fit and the apply then run on the stretched values
        (applied on the fly; the stretched planes are never written).

        ``stretch_scope`` says over which pixels the percentiles are taken.  "granule" (default): per image, and a
        global fit (``synthesize_sharded``, ``exchange=`` / ``allreduce=True``) with a stretch raises ``ValueError``.
        "fit": over exactly the pixels the fit is taken over — one granule, each tile of ``synthesize_tiles``, or the
        union of every granule / slab on every rank of a global fit (exact: np.percentile of the concatenation, the
        same limits on every rank)."""
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
        if self.stretch is not None:
            fm = self.stretch_mask(bands, s2_ref, valid, fit_mask, groups=groups)
            xl, yl = self.stretch_limits([(bands, s2_ref, fm)], reduce, groups=groups)
            mom, fm = kernels.fit_moments(bands, s2_ref, fm, self.deg, groups=groups, mask_given=True,
                                          x_stretch=xl, y_stretch=yl, exchange=exchange)
            return mom, fm, xl, yl
        if self.y_finite:
            mom, fm = kernels.fit_moments(bands, s2_ref, valid, self.deg, groups=groups, gate_k=self.gate_k,
                                          gate_gt=0.0, y_finite=True, exchange=exchange)
        else:
            mom, fm = kernels.fit_moments(bands, s2_ref, fit_mask, self.deg, groups=groups, mask_given=True,
                                          exchange=exchange)
        return mom, fm, None, None

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

    def moments(self, bands, s2_ref, fit_mask, mask_rows="auto"):
        return kernels.poly_moments(bands, s2_ref, fit_mask, self.deg, mask_rows=mask_rows)

    # ------------------------------------------------------------------ one granule
    def synthesize(self, raw: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor, s2_ref: torch.Tensor, *,
                   transpose_raw_yx: bool = False, materialize_ortho: bool = False, group=None,
                   allreduce: bool = False, bands_out=None, matched_out=None, exchange=None,
                   raw_row0: int = 0, raw_rows_total: Optional[int] = None) -> PairResult:
        """raw [Hr, Wr, B] f32, GLT planes [Ho, Wo] int32, s2_ref [K, Ho, Wo] f32 — all CUDA tensors.
        Three launches (+ the moment finalize): glt_srf, fit_moments, poly_solve_apply.
        Global fit across ranks: ``exchange`` (a ``dist.PeerExchange``: moments travel over NVLink peer memory
        inside the finalize / solve kernels) or ``allreduce=True`` (one NCCL all-reduce between the two)."""
        global_fit = (exchange is not None and exchange.world > 1) or (allreduce and hdist.world()[1] > 1)
        if global_fit:
            self._no_global_stretch("exchange= / allreduce=True")
        fm = torch.empty(glt_x.shape, dtype=torch.bool, device=raw.device)
        bands, valid, diag, ortho = self.bands_from_raw(raw, glt_x, glt_y, transpose_raw_yx=transpose_raw_yx,
                                                        materialize_ortho=materialize_ortho, bands_out=bands_out,
                                                        fit_mask_out=fm, raw_row0=raw_row0,
                                                        raw_rows_total=raw_rows_total)
        ex = exchange.next() if exchange is not None and exchange.world > 1 else None
        reduce = self._global_reduce(group) if global_fit else None
        mom, fm, xl, yl = self.fit(bands, s2_ref, valid, fm, exchange=ex, reduce=reduce)
        if allreduce and ex is None:
            hdist.allreduce_moments(mom, group)
        lo, hi = self.clip if self.clip is not None else (1.0, 0.0)
        gmom = torch.empty_like(mom) if ex is not None else None
        coeffs, matched = kernels.poly_solve_apply(bands, mom, fm, self.deg, min_count=self.min_count, lo=lo, hi=hi,
                                                   out=matched_out, x_stretch=xl, exchange=ex, moments_out=gmom)
        if gmom is not None:
            mom = gmom
        return PairResult(bands, matched, coeffs.view(self.K, self.deg + 1), valid, fm.view(valid.shape), diag,
                          mom.view(self.K, -1), ortho, self.band_names, xl, yl)

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
        import numpy as np

        if isinstance(raw, np.ndarray):
            raw = torch.from_numpy(raw)
        d0, d1 = int(raw.shape[0]), int(raw.shape[1])
        Hr, Wr = (d1, d0) if transpose_raw_yx else (d0, d1)
        with torch.cuda.device(self.device):
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
            res = self.synthesize(win, glt_x, glt_y, s2_ref, transpose_raw_yx=transpose_raw_yx, raw_row0=lo,
                                  raw_rows_total=d0, **kw)
            outside = int(res.diag[3])
            if outside:
                raise RuntimeError(f"{outside} valid GLT entries fell outside the staged raw rows [{lo}, {hi})")
        res.diag = res.diag[:3]
        res.raw_rows = (lo, hi)
        return res

    # ------------------------------------------------------------------ a batch of equal tiles
    def synthesize_tiles(self, raw_tiles: torch.Tensor, glt_x: torch.Tensor, glt_y: torch.Tensor,
                         s2_ref: torch.Tensor) -> PairResult:
        """Tile batch (tiles_helpers shape contract): raw_tiles [T, h, w, B], GLT planes [T, h, w] with
        per-tile 1-based indices, s2_ref [K, T, h, w].  One launch per stage; T*K independent fits.
        The tiles are stacked along rows; the kernel itself offsets tile t's GLT rows by t*h and keeps an entry that
        points past its own tile out of bounds (hsr_raw_view_t.batch_*), so the GLT is used as delivered."""
        T, h, w, B = raw_tiles.shape
        gy = glt_y.reshape(T * h, w)
        gx = glt_x.reshape(T * h, w)
        raw = raw_tiles.reshape(T * h, w, B)
        fm = torch.empty(gx.shape, dtype=torch.bool, device=raw.device)
        bands, valid, diag, _ = self.bands_from_raw(raw, gx, gy, fit_mask_out=fm, tile_rows=(h, h))   # [K, T*h, w]
        diag = diag[:3]
        mom, fm, xl, yl = self.fit(bands, s2_ref, valid, fm.view(T, h * w), groups=T)
        lo, hi = self.clip if self.clip is not None else (1.0, 0.0)
        coeffs, matched = kernels.poly_solve_apply(bands, mom, fm, self.deg, groups=T, min_count=self.min_count,
                                                   lo=lo, hi=hi, x_stretch=xl)
        return PairResult(bands.view(self.K, T, h, w), matched.view(self.K, T, h, w), coeffs, valid.view(T, h, w),
                          fm.view(T, h, w), diag, mom, None, self.band_names, xl, yl)

    # ------------------------------------------------------------------ many granules, one global fit
    def synthesize_sharded(self, granules: Sequence[dict], *, group=None, exchange=None) -> List[PairResult]:
        """Granules owned by THIS rank (dicts with raw, glt_x, glt_y, s2_ref) — BASELINE configs[3]; the fit is
        GLOBAL: the local moments are summed in a fixed order (``kernels.moments_sum``), summed across ranks once —
        over NVLink peer memory when ``exchange`` (a ``dist.PeerExchange``) is given, else one all-reduce (NCCL /
        gloo) — and solved redundantly.  A rank that was dealt no granule still takes part in the exchange.
        With ``stretch_scope="fit"`` the stretch limits are the percentiles of every granule on every rank (their
        histograms are summed over ``group`` with ``dist.all_reduce`` also when the moments go through ``exchange``)."""
        self._no_global_stretch("synthesize_sharded")
        stage = []
        for g in granules:
            fm = torch.empty(g["glt_x"].shape, dtype=torch.bool, device=self.device)
            bands, valid, diag, _ = self.bands_from_raw(g["raw"], g["glt_x"], g["glt_y"],
                                                        transpose_raw_yx=g.get("transpose_raw_yx", False),
                                                        fit_mask_out=fm)
            if self.stretch is not None:
                fm = self.stretch_mask(bands, g["s2_ref"], valid, fm)
            stage.append((bands, valid, diag, fm, g["s2_ref"]))
        xl = yl = None
        if self.stretch is not None:
            xl, yl = self.stretch_limits([(s[0], s[4], s[3]) for s in stage], self._global_reduce(group))
        moms = []
        for i, (bands, valid, diag, fm, s2_ref) in enumerate(stage):
            if self.stretch is not None:
                mom, _ = kernels.fit_moments(bands, s2_ref, fm, self.deg, mask_given=True, x_stretch=xl, y_stretch=yl)
            else:
                mom, fm, _, _ = self.fit(bands, s2_ref, valid, fm)
            moms.append(mom.view(self.K, -1))
            stage[i] = (bands, valid, diag, fm)
        ex = exchange.next() if exchange is not None and exchange.world > 1 else None
        like = torch.empty((self.K, 3 * self.deg + 2), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            mom = kernels.moments_sum(moms, like=like, exchange=ex)
        if ex is None:
            hdist.allreduce_moments(mom, group)
        lo, hi = self.clip if self.clip is not None else (1.0, 0.0)
        out = []
        if ex is not None and not stage:
            # nothing to apply here, but the exchange must be consumed (the slot parity protocol lets a rank run at
            # most one epoch ahead of its own consumption)
            x0 = torch.zeros((self.K, 1), dtype=torch.float32, device=self.device)
            m0 = torch.zeros(1, dtype=torch.uint8, device=self.device)
            kernels.poly_solve_apply(x0, mom, m0, self.deg, min_count=self.min_count, lo=lo, hi=hi, exchange=ex)
        for i, (bands, valid, diag, fm) in enumerate(stage):
            if i == 0 and ex is not None:
                gmom = torch.empty_like(mom)
                coeffs, matched = kernels.poly_solve_apply(bands, mom, fm, self.deg, min_count=self.min_count, lo=lo,
                                                           hi=hi, x_stretch=xl, exchange=ex, moments_out=gmom)
                mom = gmom.view(self.K, -1)
            else:
                coeffs, matched = kernels.poly_solve_apply(bands, mom, fm, self.deg, min_count=self.min_count, lo=lo,
                                                           hi=hi, x_stretch=xl)
            out.append(PairResult(bands, matched, coeffs.view(self.K, self.deg + 1), valid, fm.view(valid.shape), diag,
                                  mom, None, self.band_names, xl, yl))
        return out


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
