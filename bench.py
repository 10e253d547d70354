#!/usr/bin/env python
"""bench.py — EMIT -> S2 pair synthesis (GLT ortho + SRF + polyfit + apply) on synthetic granules.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--config granule|ortho_srf|tiles|shards|mosaic] [--dump-outputs DIR]

Default (`--config granule`) = BASELINE.json configs[1], the configuration the metric is quoted on: one "step" = one pass
of the hot path over one synthetic EMIT-granule-shaped cube per GPU (raw 1280 x 1242 x 285 fp32, 25-degree GLT ->
1685 x 1667 ortho grid, 12 S2 bands, degree-2 fit against a synthetic S2 reference, apply).  With N > 1 every rank owns
its own granule (weak scaling) and the fit is global (moments summed over the ranks).  Prints ONE JSON line (rank 0).

Timed regions
  value   device-resident: inputs already in HBM, CUDA events, barrier + synchronize on both sides, max over ranks.
          The 1.8 GB raw cube is >> the 126 MB L2 and two input sets alternate, so no explicit L2 flush.
  e2e     the same pass through the public host-side API (HostGranuleStream) with HOST (pinned) buffers: every step
          copies the raw cube, GLT planes and S2 reference host->device and the matched planes, coefficients and valid
          mask device->host inside the timed region.  The results of the last step are compared BIT FOR BIT with a
          device-resident pass over the same inputs; the pinned host->device ceiling of the box is measured beside it.
  roofline  the fused glt_srf kernel, timed per launch with CUDA events; achieved = algorithmic bytes / duration.
  variants  (granule config) the reference script's real order with the shared percentile stretch between SRF and fit
          (s2_emit/poly_regression.py:126-127) and the script's degree 4 — reported beside, never instead of, the headline.
  cpu_baseline  the numpy oracle (a port of the reference's numpy path; the reference cannot travel to the GPU box) on the
          640 x 621 quarter granule of BASELINE.md section 3, one process, whole-cube evaluation as the reference does.
--impl reference times that oracle port on all host cores (row-split over processes), a bounded row sample per step.

The other configs are BASELINE.json's parity-test cases made driver-visible: ortho_srf = configs[0], tiles = configs[2]
(512 paired 256 x 256 tiles), shards = configs[3] as written (64 granules, seeds 100..163, round-robin, ONE global fit,
strong scaling), mosaic = configs[4] (8192 x 8192 ortho grid in row slabs, per-slab raw windows).
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "EMIT->S2 synth Mpix/s (GLT ortho+SRF+polyfit)"
UNIT = "Mpix/s"
THETA = 25.0
DEG = 2
QUARTER_RAW = (640, 621)          # BASELINE.md section 3: the quarter granule of the CPU baseline


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _env_knobs():
    """HSR_* variables in the environment.  The product library reads none (they exist only in the -DHSR_EXPERIMENTS
    build that HSR_B200_EXPERIMENTAL_LIB selects), and a benchmark must not run with that build."""
    return sorted(k for k in os.environ if k.startswith("HSR_"))


class ClockSampler(threading.Thread):
    """Polls SM clock + throttle reasons through NVML while the timed region runs."""

    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.ok = index, [], set(), None, False
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        if not self.ok:
            return
        try:
            self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            r = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for bit, name in self.BITS.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self.sample()
            time.sleep(0.001)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _physical_index(local_index):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_index])
        except Exception:
            return local_index
    return local_index


# ------------------------------------------------------------------------------------ CPU arms
def _cpu_inputs(seed, block, raw_hw=None):
    """Host inputs for an ortho block (r0, r1, c0, c1) of a synthetic granule (same generators, numpy).
    Only the raw patch the block references is generated (the full cube is 1.8 GB)."""
    from hsr_b200 import synthetic
    from hsr_b200.s2_emit.srf import synthetic_s2_srf

    Hr, Wr, B = synthetic.GRANULE_RAW_SHAPE
    if raw_hw is not None:
        Hr, Wr = raw_hw
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    gx, gy = synthetic.rotation_glt(Hr, Wr, THETA)
    r0, r1, c0, c1 = block
    gxs, gys = gx[r0:r1, c0:c1], gy[r0:r1, c0:c1]
    ok = (gxs > 0) & (gys > 0)
    if ok.any():
        y_lo, y_hi = int(gys[ok].min()) - 1, int(gys[ok].max())
        x_lo, x_hi = int(gxs[ok].min()) - 1, int(gxs[ok].max())
    else:
        y_lo, y_hi, x_lo, x_hi = 0, 1, 0, 1
    raw = synthetic.raw_cube_spectra_np((y_hi - y_lo, x_hi - x_lo, B), seed=seed, good=good)
    gys = np.where(ok, gys - y_lo, 0).astype(np.int32)
    gxs = np.where(ok, gxs - x_lo, 0).astype(np.int32)
    return raw, gxs, gys, w, good, synthetic_s2_srf()


def _cpu_ortho_srf(raw, gx, gy, w, good, table):
    """apply_glt -> pseudo_s2_srf_integral, restated in oracle/ (WHOLE-cube evaluation per band, as the reference:
    no row slabs — the four cube-sized float64 temporaries of synth.py:41 are part of what is timed)."""
    from oracle import glt as oglt
    from oracle import srf as osrf

    ortho, valid, _ = oglt.glt_ortho(raw, gx, gy)
    ps = osrf.pseudo_s2_srf_integral(ortho, w, table, good, rows_per_slab=max(1, ortho.shape[0]))
    x = np.stack([p for p in ps.values() if p is not None]).astype(np.float32)
    return x, valid


def _cpu_fit_apply(x, valid, s2=None):
    """np.polyfit per band over all valid pixels -> apply_poly_rgb-style Horner + mask + clip."""
    from hsr_b200 import synthetic
    from oracle import poly as opoly

    if s2 is None:
        s2 = synthetic.s2_reference_np(x, seed=1)
    fm = opoly.fit_mask(x, valid, 0, 0.0)
    coeffs = opoly.polyfit_paired(x, s2, fm, DEG, min_count=200)
    matched = opoly.apply_poly_planes(x, coeffs, fm)
    return matched.shape[1] * matched.shape[2]


def _cpu_pass(raw, gx, gy, w, good, table):
    x, valid = _cpu_ortho_srf(raw, gx, gy, w, good, table)
    return _cpu_fit_apply(x, valid)


_JOBS = []   # filled before the worker pool forks, so the inputs are shared, not pickled


def _cpu_worker(i):
    import warnings
    warnings.simplefilter("ignore")
    return _cpu_ortho_srf(*_JOBS[i])


def cpu_baseline():
    """BASELINE.md section 3: the 640 x 621 quarter granule ONCE, one process, through the oracle port with the
    reference's whole-cube evaluation; raw seconds and Mpix/s both stated."""
    import warnings

    from hsr_b200 import synthetic
    warnings.simplefilter("ignore")
    Hq, Wq = QUARTER_RAW
    gx, _ = synthetic.rotation_glt(Hq, Wq, THETA)
    Ho, Wo = gx.shape
    inputs = _cpu_inputs(0, (0, Ho, 0, Wo), raw_hw=QUARTER_RAW)
    t0 = time.perf_counter()
    npx = _cpu_pass(*inputs)
    dt = time.perf_counter() - t0
    return {"value": npx / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port", "seconds": round(dt, 2),
            "pixels": npx,
            "sample": f"quarter granule (BASELINE.md section 3): raw {Hq}x{Wq}x285 f32 + {THETA:g}deg GLT -> {Ho}x{Wo} ortho grid "
                      f"({npx} px), ortho + SRF(12 bands, whole-cube float64 evaluation as s2_emit/synth.py:41) + polyfit(deg "
                      f"{DEG}) + apply, numpy oracle port of the reference path, 1 process, timed once: {dt:.1f} s"}


def run_reference(args):
    """--impl reference: the oracle port on all host cores.  Row-split over one process per core (BASELINE.md section 3,
    "reference x N processes (row-split)"): per step every process does ortho + SRF of its own block of full-width
    ortho rows of the quarter granule (not cache-resident: ~45 MB per float64 temporary), the parent fits and applies
    over all of them."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import warnings

    from hsr_b200 import synthetic
    warnings.simplefilter("ignore")
    cores = os.cpu_count() or 1
    Hq, Wq = QUARTER_RAW
    gx, _ = synthetic.rotation_glt(Hq, Wq, THETA)
    Ho, Wo = gx.shape
    rows = 24                                          # full-width ortho rows per process and step (~2 s of numpy)
    first = max(0, (Ho - rows * cores) // 2)           # centred: these rows cross the whole swath
    for i in range(cores):
        r0 = min(Ho - rows, first + i * rows)
        _JOBS.append(_cpu_inputs(0, (r0, r0 + rows, 0, Wo), raw_hw=QUARTER_RAW))
    ctx = mp.get_context("fork")
    times = []
    npx = 0
    with ctx.Pool(cores) as pool:
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            parts = pool.map(_cpu_worker, range(cores), chunksize=1)
            x = np.concatenate([p[0] for p in parts], axis=1)
            valid = np.concatenate([p[1] for p in parts], axis=0)
            npx = _cpu_fit_apply(x, valid)
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = npx / (ms / 1e3) / 1e6
    sample = (f"{cores} processes x {rows} full-width ortho rows ({npx} px per step) of the quarter granule "
              f"(raw {Hq}x{Wq}x285, {Ho}x{Wo} ortho grid), row-split: ortho + SRF(12 bands, float64) per process, "
              f"polyfit(deg {DEG}) + apply over all rows in the parent; numpy oracle port of the reference path")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1]: synthetic EMIT granule 1280x1242x285 f32 + 25deg GLT -> ortho + SRF "
                               "(12 S2 bands) + degree-2 polyfit + apply; bounded row sample of the quarter granule per step",
                   "l2": "n/a (CPU)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ GPU arm: helpers
def graph_node_counts(graph):
    """(kernel, memset, other) nodes of a captured torch.cuda.CUDAGraph (created with keep_graph=True), read with the
    driver API — the launches one replay performs, counted, not assumed."""
    try:
        cu = ctypes.CDLL("libcuda.so.1")
        g = ctypes.c_void_p(graph.raw_cuda_graph())
        n = ctypes.c_size_t(0)
        if cu.cuGraphGetNodes(g, None, ctypes.byref(n)) != 0:
            return None
        nodes = (ctypes.c_void_p * max(1, n.value))()
        if cu.cuGraphGetNodes(g, nodes, ctypes.byref(n)) != 0:
            return None
        kern = mset = other = 0
        for i in range(n.value):
            t = ctypes.c_int(-1)
            cu.cuGraphNodeGetType(ctypes.c_void_p(nodes[i]), ctypes.byref(t))
            if t.value == 0:
                kern += 1
            elif t.value == 2:
                mset += 1
            else:
                other += 1
        return kern, mset, other
    except Exception:
        return None


class Ctx:
    """What every GPU config needs: ranks, device, the synthesizer."""

    def __init__(self, args, deg=DEG, stretch=None):
        import torch
        import torch.distributed as dist

        from hsr_b200 import dist as hdist
        from hsr_b200 import synthetic
        from hsr_b200.pipeline import PairSynthesizer
        from hsr_b200.s2_emit.srf import synthetic_s2_srf

        self.torch, self.dist, self.hdist, self.synthetic = torch, dist, hdist, synthetic
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: hsr_b200 has no CPU path (use --impl reference for the CPU arm)")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL prints its banner there)
        self.rank, self.world, self.device = hdist.init_from_env()
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        self.multi = self.world > 1
        self.w = synthetic.emit_wavelengths()
        self.good = synthetic.good_band_mask(self.w)
        self.table = synthetic_s2_srf()
        self.PairSynthesizer = PairSynthesizer
        self.ps = PairSynthesizer(self.w, self.table, self.good, deg=deg, device=self.device, stretch=stretch)
        self.K = self.ps.K
        self.sampler = ClockSampler(_physical_index(self.device.index or 0))

    def barrier(self):
        if self.multi:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.device)
        if self.multi:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def finish(self, px=None):
        if self.multi:
            self.dist.barrier()
            self.torch.cuda.synchronize()
            if px is not None:
                px.close()
            self.dist.destroy_process_group()


def timed_loop(ctx, run, steps):
    """barrier + sync | EXACTLY `steps` calls of run(i) between two CUDA events | barrier + sync; ms total (this rank)."""
    torch = ctx.torch
    ctx.barrier()
    ctx.sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        run(i)
    t1.record()
    ctx.sampler.sample()
    ctx.barrier()
    ctx.sampler.stop()
    return t0.elapsed_time(t1)


def capture(ctx, fn):
    """fn captured into a CUDA graph (warm-up on a side stream first); returns (graph, node counts, fn's return value,
    whose tensors every replay rewrites in place)."""
    torch = ctx.torch
    side = torch.cuda.Stream(ctx.device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    try:
        g = torch.cuda.CUDAGraph(keep_graph=True)
    except TypeError:                                  # older torch: no node introspection
        g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    counts = graph_node_counts(g)
    try:
        g.instantiate()
    except Exception:
        pass
    return g, counts, out


DUMP_SAMPLE_PX = 1 << 18


def dump_outputs(out_dir, outputs, grid_hw):
    """--dump-outputs: each output as out_dir/<name>.npy (float64 stays float64, everything else becomes float32).
    Per-pixel outputs ([K, Ho, Wo] planes, [Ho, Wo] masks) are kept at the same DUMP_SAMPLE_PX ortho pixels in every
    array and every run (flat indices drawn by numpy's default_rng(0), sorted): the full planes are 135 MB each."""
    import torch

    Ho, Wo = grid_hw
    idx = np.sort(np.random.default_rng(0).choice(Ho * Wo, size=min(Ho * Wo, DUMP_SAMPLE_PX), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        if tuple(t.shape[-2:]) == (Ho, Wo):
            t = t[..., torch.from_numpy(idx // Wo).to(t.device), torch.from_numpy(idx % Wo).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def base_line(ctx, args, value, ms_per_step, scaling, config):
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "env_knobs": _env_knobs()}


# ------------------------------------------------------------------------------------ configs[1] (default) / configs[0]
def run_granule(args, ortho_srf_only=False):
    ctx = Ctx(args)
    torch, hdist, synthetic, ps = ctx.torch, ctx.hdist, ctx.synthetic, ctx.ps
    from hsr_b200 import kernels
    rank, world, device, multi, K = ctx.rank, ctx.world, ctx.device, ctx.multi, ctx.K

    Hr, Wr, B = synthetic.GRANULE_RAW_SHAPE
    gx_np, gy_np = synthetic.rotation_glt(Hr, Wr, THETA)
    gx = torch.from_numpy(gx_np).to(device)
    gy = torch.from_numpy(gy_np).to(device)
    Ho, Wo = gx_np.shape
    n_o = Ho * Wo
    n_v = int(((gx_np != 0) & (gy_np != 0)).sum())
    # TWO input sets (raw cube + Sentinel-2 planes, different seeds) alternate between the timed steps, so that no step
    # finds in L2 what the previous one read
    sets = []
    for si in range(2):
        raw_i = synthetic.raw_cube_spectra_torch((Hr, Wr, B), seed=(100 + rank if multi else 0) + 1000 * si, device=device,
                                                 good=ctx.good)
        bands0, _, _, _ = ps.bands_from_raw(raw_i, gx, gy)
        s2_i = kernels.alloc_planes(K, (Ho, Wo), device)     # plane stride padded to 128 B: 16-byte loads in the fit
        s2_i.copy_(synthetic.s2_reference_torch(bands0, seed=1 + rank + 1000 * si))
        del bands0
        sets.append((raw_i, s2_i))

    # preallocated outputs: the timed region launches kernels of libhsr_b200.so only (no torch kernel, no memset)
    bands = kernels.alloc_planes(K, (Ho, Wo), device)
    matched = kernels.alloc_planes(K, (Ho, Wo), device)
    fit_mask = torch.empty((Ho, Wo), dtype=torch.bool, device=device)
    valid_buf = torch.empty((Ho, Wo), dtype=torch.bool, device=device)
    lo, hi = ps.clip
    ev_pairs = []
    px = None
    if multi and args.collective == "peer" and not ortho_srf_only:
        try:
            px = hdist.PeerExchange(device=device)
        except hdist.PeerExchangeUnavailable as e:     # raised on every rank alike: all of them fall back to NCCL
            if rank == 0:
                print(f"[bench] peer exchange unavailable ({e}); using the NCCL all-reduce", file=sys.stderr)
            args.collective = "nccl"

    def step(record=False, si=0, syn=ps, deg=DEG, collective=True):
        raw, s2 = sets[si]
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        b, valid, _, _ = syn.bands_from_raw(raw, gx, gy, bands_out=bands, fit_mask_out=fit_mask, valid_out=valid_buf,
                                            want_diag=False)
        if record:
            e1.record()
            ev_pairs.append((e0, e1))
        if ortho_srf_only:
            return None
        ex = px.next() if (px is not None and collective) else None
        mom, fm, xl, _ = syn.fit(b, s2, valid, fit_mask, exchange=ex)
        if multi and px is None and args.collective == "nccl" and collective:
            hdist.allreduce_moments(mom)
        coeffs, _ = kernels.poly_solve_apply(b, mom, fm, deg, min_count=syn.min_count, lo=lo, hi=hi, out=matched,
                                             exchange=ex, x_stretch=xl)
        return coeffs

    for i in range(args.warmup):
        step(si=i & 1)
    ctx.barrier()
    graphs, counts = None, None
    coeffs_out = [None, None]      # the coefficients each input set's step returns (rewritten by every replay)
    if not args.no_graph and (not multi or px is not None or ortho_srf_only):
        # the step's launches captured once per input set and replayed: same kernels, same arguments, ~1 us between
        # dependent kernels instead of ~3 us
        graphs = []
        for si in range(2):
            g, c, coeffs_out[si] = capture(ctx, lambda si=si: step(si=si))
            graphs.append(g)
            counts = c if c is not None else counts
        for i in range(4):
            graphs[i & 1].replay()
        torch.cuda.synchronize()

    def eager_step(i):
        coeffs_out[i & 1] = step(record=True, si=i & 1)

    ms_total = timed_loop(ctx, (lambda i: graphs[i & 1].replay()) if graphs is not None else eager_step, args.steps)
    if args.dump_outputs and rank == 0:
        # the last timed step's outputs, before the steps below overwrite the shared buffers
        outputs = {"bands": bands, "valid": valid_buf, "fit_mask": fit_mask}
        if not ortho_srf_only:
            outputs.update(matched=matched, coeffs=coeffs_out[(args.steps - 1) & 1])
        dump_outputs(args.dump_outputs, outputs, (Ho, Wo))
    if graphs is not None:      # kernel time of the fused gather, from eager steps (events cannot be read from a replay)
        for i in range(30):
            step(record=True, si=i & 1)
        ctx.barrier()
        del ev_pairs[:10]
    srf_ms = float(np.mean([a.elapsed_time(b) for a, b in ev_pairs]))
    ms_total, srf_ms = ctx.max_over_ranks([ms_total, srf_ms])
    ms_per_step = ms_total / args.steps
    value = world * n_o / (ms_per_step / 1e3) / 1e6
    per_step_kernels = counts[0] if counts else (1 if ortho_srf_only else 4)

    # ---------------------------------------------------------------- variants (reported beside the headline)
    variants = {}
    if not ortho_srf_only and not args.no_variants and not multi:
        def time_variant(name, syn, deg, note):
            for i in range(3):
                step(si=i & 1, syn=syn, deg=deg)
            torch.cuda.synchronize()
            try:
                gs = [capture(ctx, lambda si=si: step(si=si, syn=syn, deg=deg)) for si in range(2)]
                run, nodes = (lambda i: gs[i & 1][0].replay()), gs[0][1]
            except Exception:
                torch.cuda.synchronize()
                run, nodes = (lambda i: step(si=i & 1, syn=syn, deg=deg)), None
            for i in range(4):
                run(i)
            torch.cuda.synchronize()
            n = max(10, min(args.steps, 50))
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n):
                run(i)
            b_.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b_) / n
            variants[name] = {"ms_per_step": ms, "value": n_o / (ms / 1e3) / 1e6, "unit": UNIT, "steps": n,
                              "kernels_per_step": nodes[0] if nodes else None, "what": note}

        time_variant("stretch_2_98", ctx.PairSynthesizer(ctx.w, ctx.table, ctx.good, deg=DEG, device=device, stretch=(2, 98)),
                     DEG, "the reference script's order (s2_emit/poly_regression.py:126-127): shared 2/98 percentile stretch of both "
                          "images (exact radix select) between SRF and fit, fit and apply on the stretched values")
        time_variant("deg4", ctx.PairSynthesizer(ctx.w, ctx.table, ctx.good, deg=4, device=device), 4,
                     "degree 4, the reference script's own degree (poly_regression.py:133)")

    e2e = None
    if not ortho_srf_only:
        # ---------------------------------------------------------------- e2e: host buffers in, host results out
        from hsr_b200.pipeline import HostGranuleStream

        raw, s2 = sets[0]
        del bands, matched
        hs = HostGranuleStream(ps, (Hr, Wr, B), (Ho, Wo), depth=2, allreduce=multi, exchange=px)
        stride = hs.stride
        h_raw = torch.empty((Hr, Wr, B), dtype=torch.float32, pin_memory=True)
        h_raw.copy_(raw)
        h_gx, h_gy = torch.from_numpy(gx_np).pin_memory(), torch.from_numpy(gy_np).pin_memory()
        h_s2 = torch.zeros((K, stride), dtype=torch.float32, pin_memory=True)
        h_s2[:, :n_o].copy_(s2.reshape(K, n_o))
        outs = [hs.host_buffers() for _ in range(2)]
        h2d = h_raw.numel() * 4 + h_gx.numel() * 4 + h_gy.numel() * 4 + h_s2.numel() * 4
        d2h = outs[0]["matched"].numel() * 4 + outs[0]["valid"].numel() + outs[0]["coeffs"].numel() * 8
        del raw, s2, sets
        torch.cuda.empty_cache()

        # the box's pinned host->device ceiling, all ranks copying at once (what bounds e2e): the raw cube alone, 3 times
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        hs.slots[0]["raw"].copy_(h_raw, non_blocking=True)
        ctx.barrier()
        c0.record()
        for _ in range(3):
            hs.slots[0]["raw"].copy_(h_raw, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        h2d_peak = 3 * h_raw.numel() * 4 / (c0.elapsed_time(c1) / 1e3) / 1e9

        e2e_steps = max(3, min(args.steps, 10))
        for i in range(max(2, min(args.warmup, 3))):
            hs.submit(h_raw, h_gx, h_gy, h_s2, outs[i % 2])
        hs.drain()
        ctx.barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(e2e_steps):
            hs.submit(h_raw, h_gx, h_gy, h_s2, outs[i % 2])
        hs.drain()
        t1.record()
        ctx.barrier()
        e2e_ms, neg_peak = ctx.max_over_ranks([t0.elapsed_time(t1) / e2e_steps, -h2d_peak])
        h2d_peak_min = -neg_peak
        e2e_value = world * n_o / (e2e_ms / 1e3) / 1e6
        # the e2e results against a device-resident pass over the same inputs: every output bit for bit
        last = outs[(e2e_steps - 1) % 2]
        sl = hs.slots[0]
        sl["raw"].copy_(h_raw)
        sl["s2"].copy_(h_s2[:, :n_o].view(K, Ho, Wo))
        ref = ps.synthesize(sl["raw"], gx, gy, sl["s2"], allreduce=multi and px is None, exchange=px)
        torch.cuda.synchronize()
        same = (torch.equal(last["matched"][:, :n_o].contiguous().view(torch.int32),
                            ref.matched.reshape(K, n_o).cpu().view(torch.int32))
                and torch.equal(last["valid"], ref.valid.cpu())
                and torch.equal(last["coeffs"].view(torch.int64), ref.coeffs.cpu().view(torch.int64)))
        if px is not None:
            px.check()
        if ctx.max_over_ranks([0.0 if same else 1.0])[0] != 0.0:
            raise SystemExit("bench.py: the end-to-end results differ from the device-resident pass over the same inputs")
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": e2e_ms, "steps": e2e_steps,
               "results_checked": "matched planes, valid mask and coefficients of the last e2e step are bit-identical to a "
                                  "device-resident pass over the same inputs",
               "h2d_peak_gbs": h2d_peak_min, "h2d_achieved_gbs": h2d / (e2e_ms / 1e3) / 1e9,
               "frac_of_h2d_peak": h2d / (e2e_ms / 1e3) / 1e9 / h2d_peak_min,
               "h2d_peak_how": f"pinned cudaMemcpyAsync of the 1.8 GB raw cube, 3 times, {world} rank(s) copying at once, "
                               "slowest rank (per-rank GB/s)",
               "api": "hsr_b200.pipeline.HostGranuleStream (pinned host buffers; H2D / compute / D2H on "
                      "three streams, two device slots)"}

    if rank == 0:
        peak, peak_src = _peaks()
        algo = n_v * B * 4 + n_o * 8 + n_o * K * 4 + 2 * n_o   # glt_srf: raw read + GLT + K planes + valid + fit mask
        achieved = algo / (srf_ms / 1e3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "glt_srf_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        # + moments (x, y planes, fit mask) + solve_apply (x, mask in, matched out)
        total_algo = algo if ortho_srf_only else algo + (2 * n_o * K * 4 + n_o) + (2 * n_o * K * 4 + n_o)
        name = ("configs[0]: synthetic EMIT granule 1280x1242x285 f32 + 25deg GLT -> 1685x1667 ortho + SRF (12 S2 bands), "
                "fused (the ortho cube is not materialised)") if ortho_srf_only else (
            "configs[1]: synthetic EMIT granule 1280x1242x285 f32 + 25deg GLT -> "
            "1685x1667 ortho + SRF (12 S2 bands) + degree-2 polyfit vs synthetic S2 + apply"
            + ("; one granule per rank, moments summed over the ranks" if multi else ""))
        config = {"workload": name, "pixels_per_step_per_gpu": n_o, "valid_fraction": round(n_v / n_o, 4), "srf_bands": K,
                  "deg": DEG, "l2": "inputs exceed the 126 MB L2 (1.81 GB raw cube + 0.13 GB S2 planes per set) and two input sets "
                                    "alternate between steps; no explicit flush",
                  "parallelism": f"dp{world}",
                  "launch": (f"the step ({per_step_kernels} kernels) captured once per input set into a CUDA graph and replayed"
                             if graphs is not None else f"{per_step_kernels} kernel launches per step"),
                  "collective": ("none (single GPU)" if not multi else
                                 "none (no fit in this config)" if ortho_srf_only else
                                 "moments over NVLink peer memory (CUDA IPC), fused into the finalize / solve kernels"
                                 if px is not None else "NCCL all-reduce of the fp64 moments"
                                 if args.collective == "nccl" else "NONE (diagnostic run: per-rank fits, not a result)")}
        line = base_line(ctx, args, value, ms_per_step, "weak", config)
        line["roofline"] = {"kernel": "glt_stream_kernel<SRF> (fused GLT gather + SRF)", "bound": "hbm",
                            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": traffic, "traffic_source": "ncu --set full of this kernel on this workload, "
                                                                  "profiles/glt_srf_traffic.json (regenerated by profiles/run_gpu.sh)",
                            "peak_source": peak_src, "algorithmic_bytes": algo,
                            "kernel_ms": srf_ms, "step_frac_of_peak": total_algo / (ms_per_step / 1e3) / 1e9 / peak,
                            "frac_of_8TBps": achieved / 8000.0}
        if e2e is not None:
            line["e2e"] = e2e
        line["gpu_launches"] = per_step_kernels * args.steps
        line["graph_nodes_per_step"] = ({"kernel": counts[0], "memset": counts[1], "other": counts[2]} if counts else None)
        line["clocks"] = ctx.sampler.summary()
        if variants:
            line["variants"] = variants
        if not args.no_cpu and world == 1 and not ortho_srf_only:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line))
    ctx.finish(px)


# ------------------------------------------------------------------------------------ configs[2]: 512 paired tiles
def run_tiles(args):
    ctx = Ctx(args)
    torch, ps, device, K = ctx.torch, ctx.ps, ctx.device, ctx.K
    T_all, h, B = 512, 256, 285
    mine = ctx.hdist.shard_units(T_all, ctx.rank, ctx.world)       # tiles are independent: dealt round-robin, no exchange
    T = len(mine)
    g = torch.Generator(device=device).manual_seed(1234 + ctx.rank)
    raw = torch.empty((T, h, h, B), dtype=torch.float32, device=device)
    spec = 0.6 + 0.4 * torch.sin(0.02 * torch.arange(B, device=device))
    for t0 in range(0, T, 32):
        t1 = min(T, t0 + 32)
        a = torch.rand((t1 - t0, h, h, 1), generator=g, device=device) * 0.7 + 0.05
        raw[t0:t1] = a * spec + 0.02 * (torch.rand((t1 - t0, h, h, B), generator=g, device=device) - 0.5)
        del a
    ii = torch.arange(h, device=device, dtype=torch.int32)
    gy = (ii.view(1, h, 1) + 1).expand(T, h, h).contiguous()
    gx = (ii.view(1, 1, h) + 1).expand(T, h, h).contiguous()
    gx[torch.rand((T, h, h), generator=g, device=device) < 0.02] = 0          # identity + 1 with 2 % holes (SURVEY 8d-2)
    b0 = ps.synthesize_tiles(raw, gx, gy, torch.zeros((K, T, h, h), device=device)).bands
    s2 = ctx.synthetic.s2_reference_torch(b0, seed=7 + ctx.rank)
    del b0
    for _ in range(max(3, args.warmup)):
        res = ps.synthesize_tiles(raw, gx, gy, s2)
    nv = int(res.valid.sum())
    del res
    ms_total = timed_loop(ctx, lambda i: ps.synthesize_tiles(raw, gx, gy, s2), args.steps)
    (ms_total,) = ctx.max_over_ranks([ms_total])
    ms = ms_total / args.steps
    n = T_all * h * h
    npx = T * h * h
    if ctx.rank == 0:
        peak, peak_src = _peaks()
        algo = nv * B * 4 + npx * 8 + npx * K * 4 + 2 * npx + 2 * (2 * npx * K * 4 + npx)
        config = {"workload": f"configs[2]: {T_all} paired 256x256x285 tiles (38 GB of raw tiles), ortho + SRF + {T_all * K} "
                              "per-tile degree-2 fits + apply, one launch per stage; tiles dealt round-robin to the ranks",
                  "tiles_per_gpu": T, "l2": "38 GB working set >> L2", "parallelism": f"dp{ctx.world}",
                  "collective": "none (per-tile fits)"}
        line = base_line(ctx, args, n / (ms / 1e3) / 1e6, ms, "strong", config)
        line["roofline"] = {"kernel": "whole step (glt_stream<SRF> + moments + finalize + solve_apply)", "bound": "hbm",
                            "achieved": algo / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": algo / (ms / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                            "algorithmic_bytes": algo}
        line["gpu_launches"] = 4 * args.steps
        line["clocks"] = ctx.sampler.summary()
        line["peak_hbm_gb"] = torch.cuda.max_memory_allocated() / 2 ** 30
        print(json.dumps(line))
    ctx.finish()


# ------------------------------------------------------------------------------------ configs[3]: 64 granules, one fit
def run_shards(args):
    ctx = Ctx(args)
    torch, ps, device, K, synthetic, hdist = ctx.torch, ctx.ps, ctx.device, ctx.K, ctx.synthetic, ctx.hdist
    from hsr_b200 import kernels
    n_gran = args.granules
    Hr, Wr, B = synthetic.GRANULE_RAW_SHAPE
    gx_np, gy_np = synthetic.rotation_glt(Hr, Wr, THETA)
    gx, gy = torch.from_numpy(gx_np).to(device), torch.from_numpy(gy_np).to(device)
    Ho, Wo = gx_np.shape
    n_o = Ho * Wo
    mine = hdist.shard_units(n_gran, ctx.rank, ctx.world)
    free = torch.cuda.mem_get_info(device)[0]
    # per granule: raw cube + S2 planes + (per step) bands, matched, masks
    need = len(mine) * (Hr * Wr * B * 4 + 3 * K * n_o * 4 + 3 * n_o) + 2 * 2 ** 30
    if need > 0.95 * free:
        raise SystemExit(f"configs[3]: {len(mine)} granules per rank need {need / 2**30:.0f} GB, {free / 2**30:.0f} GB free "
                         f"(use more GPUs or --granules)")
    px = None
    if ctx.multi and args.collective == "peer":
        px = hdist.PeerExchange(device=device)
    granules = []
    for i in mine:                                       # seeds 100..163 (SURVEY 8d-3)
        raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), seed=100 + i, device=device, good=ctx.good)
        b0 = ps.bands_from_raw(raw, gx, gy)[0]
        s2 = kernels.alloc_planes(K, (Ho, Wo), device)
        s2.copy_(synthetic.s2_reference_torch(b0, seed=1100 + i))
        del b0
        granules.append({"raw": raw, "glt_x": gx, "glt_y": gy, "s2_ref": s2})
    torch.cuda.empty_cache()

    def step(_i=0):
        return ps.synthesize_sharded(granules, exchange=px)

    res = None
    for _ in range(max(3, args.warmup)):
        del res
        res = step()
    torch.cuda.synchronize()
    if px is not None:
        px.check()
    coeffs = res[0].coeffs.clone() if res else torch.zeros((K, DEG + 1), dtype=torch.float64, device=device)
    del res
    ms_total = timed_loop(ctx, step, args.steps)
    (ms_total,) = ctx.max_over_ranks([ms_total])
    ms = ms_total / args.steps
    if px is not None:
        px.check()
    if ctx.rank == 0:
        peak, peak_src = _peaks()
        n_v = int(((gx_np != 0) & (gy_np != 0)).sum())
        per = n_v * B * 4 + n_o * 8 + n_o * K * 4 + 2 * n_o + 2 * (2 * n_o * K * 4 + n_o)
        config = {"workload": f"configs[3]: {n_gran} synthetic EMIT granules (seeds 100..{99 + n_gran}) dealt round-robin to the "
                              "ranks, ortho + SRF per granule, ONE global degree-2 fit (local fixed-order moment sum + one "
                              "exchange per step), apply per granule",
                  "granules_per_gpu": len(mine), "l2": "1.8 GB per granule >> L2", "parallelism": f"dp{ctx.world}",
                  "collective": ("none (single GPU)" if not ctx.multi else
                                 "one exchange per step over NVLink peer memory (hsr_moments_sum_f64 publishes, the first "
                                 "solve/apply consumes)" if px is not None else "one NCCL all-reduce per step"),
                  "coeffs_band0": [float(v) for v in coeffs[0].cpu()]}
        line = base_line(ctx, args, n_gran * n_o / (ms / 1e3) / 1e6, ms, "strong", config)
        line["roofline"] = {"kernel": "whole step", "bound": "hbm", "achieved": len(mine) * per / (ms / 1e3) / 1e9,
                            "peak": peak, "unit": "GB/s", "frac": len(mine) * per / (ms / 1e3) / 1e9 / peak, "traffic": None,
                            "peak_source": peak_src, "algorithmic_bytes": len(mine) * per}
        line["gpu_launches"] = (len(mine) * 4 + 1) * args.steps
        line["clocks"] = ctx.sampler.summary()
        line["peak_hbm_gb"] = torch.cuda.max_memory_allocated() / 2 ** 30
        print(json.dumps(line))
    ctx.finish(px)


# ------------------------------------------------------------------------------------ configs[4]: 8192^2 mosaic in row slabs
def run_mosaic(args):
    ctx = Ctx(args)
    torch, ps, device, K, hdist = ctx.torch, ctx.ps, ctx.device, ctx.K, ctx.hdist
    from hsr_b200 import kernels
    Ho = Wo = 8192
    Hr = Wr = 6164
    B = 285
    th = np.deg2rad(THETA)
    # slabs balanced by WORK: the rows of the rotated swath hold very different numbers of valid pixels (the cost of a row
    # ~ valid pixels x 1140 B of spectra + 8192 x 150 B of planes / masks); equal row counts left the middle ranks with 1.3 x
    # the work of the outer ones.  Valid pixels per row from the swath's geometry (chord of the rotated square).  A nodata
    # tile costs the gather kernel ~160 ns per SM (producer latency, profiles/r2/nodata/), ~4 x its 58 B per pixel: + 170.
    rowc = np.arange(Ho, dtype=np.float64) - (Ho - 1) / 2
    xc = np.arange(Wo, dtype=np.float64) - (Wo - 1) / 2
    nvalid_row = np.empty(Ho)
    for r in range(0, Ho, 256):
        yy_ = rowc[r:r + 256, None]
        rx_ = np.rint(xc[None, :] * np.cos(th) + yy_ * np.sin(th) + (Wr - 1) / 2)
        ry_ = np.rint(-xc[None, :] * np.sin(th) + yy_ * np.cos(th) + (Hr - 1) / 2)
        nvalid_row[r:r + 256] = ((rx_ >= 0) & (rx_ < Wr) & (ry_ >= 0) & (ry_ < Hr)).sum(1)
    r0, r1 = hdist.shard_rows(Ho, ctx.rank, ctx.world, align=8, weights=nvalid_row * (B * 4.0) + Wo * (8 + 2 + 5 * ctx.K * 4.0 + 170.0))
    yy = torch.arange(r0, r1, device=device, dtype=torch.float64).view(-1, 1) - (Ho - 1) / 2
    xx = torch.arange(Wo, device=device, dtype=torch.float64).view(1, -1) - (Wo - 1) / 2
    rx = torch.round(xx * np.cos(th) + yy * np.sin(th) + (Wr - 1) / 2).to(torch.int64)
    ry = torch.round(-xx * np.sin(th) + yy * np.cos(th) + (Hr - 1) / 2).to(torch.int64)
    inside = (rx >= 0) & (rx < Wr) & (ry >= 0) & (ry < Hr)
    gx = torch.where(inside, rx + 1, torch.zeros_like(rx)).to(torch.int32)
    gy = torch.where(inside, ry + 1, torch.zeros_like(ry)).to(torch.int32)
    nv = int(inside.sum())
    del rx, ry, xx, yy, inside
    # per-slab raw window: only the raw rows this slab's GLT references are held on this GPU (SURVEY 7.3-6); the rows are
    # generated per 64-row block from the block's own seed, so every rank sees the same mosaic
    lo, hi = kernels.glt_row_range(gx, gy, Hr, Wr).tolist()
    if hi == 0:
        lo, hi = 0, 1
    raw = torch.empty((hi - lo, Wr, B), dtype=torch.float32, device=device)
    blk = 64
    for b0 in range(lo // blk * blk, hi, blk):
        g = torch.Generator(device=device).manual_seed(5000 + b0 // blk)
        rows = torch.rand((blk, Wr, B), generator=g, device=device) * 0.6
        a, b_ = max(b0, lo), min(b0 + blk, hi)
        raw[a - lo:b_ - lo] = rows[a - b0:b_ - b0]
        del rows
    n = (r1 - r0) * Wo
    px = None
    if ctx.multi and args.collective == "peer":
        px = hdist.PeerExchange(device=device)
    bands = kernels.alloc_planes(K, (r1 - r0, Wo), device)
    matched = kernels.alloc_planes(K, (r1 - r0, Wo), device)
    b0 = ps.bands_from_raw(raw, gx, gy, raw_row0=lo, raw_rows_total=Hr, bands_out=bands)[0]
    s2 = kernels.alloc_planes(K, (r1 - r0, Wo), device)
    s2.copy_(ctx.synthetic.s2_reference_torch(b0, seed=31 + ctx.rank))

    def step(_i=0):
        return ps.synthesize(raw, gx, gy, s2, raw_row0=lo, raw_rows_total=Hr, bands_out=bands, matched_out=matched,
                             exchange=px, allreduce=ctx.multi and px is None)

    for _ in range(max(3, args.warmup)):
        res = step()
    torch.cuda.synchronize()
    outside = int(res.diag[3])
    if outside:
        raise SystemExit(f"configs[4]: {outside} valid GLT entries outside the staged raw rows")
    ms_total = timed_loop(ctx, step, args.steps)
    (ms_total,) = ctx.max_over_ranks([ms_total])
    ms = ms_total / args.steps
    if px is not None:
        px.check()
    # the slabs' balance: the gather + SRF kernel alone (no exchange, so the ranks are not coupled), per rank
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(10):
        ps.bands_from_raw(raw, gx, gy, raw_row0=lo, raw_rows_total=Hr, bands_out=bands)
    e1.record()
    torch.cuda.synchronize()
    mine = torch.tensor([e0.elapsed_time(e1) / 10, float(r1 - r0), float(nv)], dtype=torch.float64, device=device)
    per_rank = [torch.zeros_like(mine) for _ in range(ctx.world)] if ctx.multi else [mine]
    if ctx.multi:
        ctx.dist.all_gather(per_rank, mine)
    hbm = ctx.max_over_ranks([torch.cuda.max_memory_allocated() / 2 ** 30])[0]
    staged = ctx.max_over_ranks([float(hi - lo)])[0]
    if ctx.rank == 0:
        peak, peak_src = _peaks()
        algo = nv * B * 4 + n * 8 + n * K * 4 + 2 * n + 2 * (2 * n * K * 4 + n)
        config = {"workload": "configs[4]: 8192x8192 ortho grid over a 6164x6164x285 raw mosaic (43.3 GB), 25deg GLT, row slabs "
                              "of the ortho grid per rank (dist.shard_rows, balanced by valid pixels per row), each rank holds only the raw rows its slab references "
                              "(hsr_raw_view_t), fused gather + SRF + ONE global degree-2 fit + apply",
                  "ortho_rows_per_gpu": r1 - r0, "raw_rows_staged_max": int(staged), "raw_rows_total": Hr,
                  "slabs": [{"rows": int(t[1]), "valid_px": int(t[2]), "gather_srf_ms": round(float(t[0]), 4)} for t in per_rank],
                  "l2": "tens of GB per rank >> L2", "parallelism": f"dp{ctx.world} (row slabs)",
                  "collective": ("none (single GPU)" if not ctx.multi else "moments over NVLink peer memory" if px is not None
                                 else "one NCCL all-reduce per step")}
        line = base_line(ctx, args, Ho * Wo / (ms / 1e3) / 1e6, ms, "strong", config)
        line["roofline"] = {"kernel": "whole step (rank 0's slab)", "bound": "hbm", "achieved": algo / (ms / 1e3) / 1e9,
                            "peak": peak, "unit": "GB/s", "frac": algo / (ms / 1e3) / 1e9 / peak, "traffic": None,
                            "peak_source": peak_src, "algorithmic_bytes": algo}
        line["gpu_launches"] = 4 * args.steps
        line["clocks"] = ctx.sampler.summary()
        line["peak_hbm_gb"] = hbm
        print(json.dumps(line))
    ctx.finish(px)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=["granule", "ortho_srf", "tiles", "shards", "mosaic"], default="granule",
                    help="granule = BASELINE configs[1] (default, the metric's configuration); ortho_srf = configs[0]; "
                         "tiles = configs[2]; shards = configs[3]; mosaic = configs[4]")
    ap.add_argument("--granules", type=int, default=64, help="--config shards: number of granules (64 = configs[3])")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-variants", action="store_true", help="skip the stretch / degree-4 variants of the granule config")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch the step's kernels one by one instead of replaying them from a CUDA graph")
    ap.add_argument("--collective", choices=["peer", "nccl", "none"], default="peer",
                    help="N > 1: moments over NVLink peer memory fused into the finalize / solve kernels (default) or one "
                         "NCCL all-reduce between them")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="granule / ortho_srf: write what the last timed step computed (rank 0's bands, matched planes, "
                         "coefficients, valid and fit masks) as DIR/<name>.npy, per-pixel outputs at a fixed sample of "
                         f"{DUMP_SAMPLE_PX} pixels; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config not in ("granule", "ortho_srf")):
        ap.error("--dump-outputs is available for --impl ours with --config granule or ortho_srf")
    knobs = _env_knobs()
    if knobs and args.impl == "ours":
        raise SystemExit(f"bench.py refuses to run with HSR_* variables set ({', '.join(knobs)}): they select or steer the "
                         "experiment build of the library (profiles/ only); unset them")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "granule":
        run_granule(args)
    elif args.config == "ortho_srf":
        run_granule(args, ortho_srf_only=True)
    elif args.config == "tiles":
        run_tiles(args)
    elif args.config == "shards":
        run_shards(args)
    else:
        run_mosaic(args)


if __name__ == "__main__":
    main()
