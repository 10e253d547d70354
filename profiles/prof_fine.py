"""Timing of the step to the Sentinel-2 10 m resolution (PairSynthesizer.matched_fine) on the granule workload of
profiles/prof_s2_grid.py: raw 1280 x 1242 x 285, 25 degree GLT, the zone 11 60 m target (1215 x 959, K = 12), factor 6
(7290 x 5754 = 41.9 Mpx per plane), deg 2 and 4, with and without the percentile stretch.  In one run, alternated:
  (a) matched_fine: fine mask -> union select over the virtual fine planes (4 count passes + 4 steps) -> fused apply;
  (b) the chain of existing kernels with the same bits: bilinear_upsample -> fit_mask(gate_k=-1) -> union select over
      the stored fine planes -> poly_solve_apply;
  (c) the percentiles alone over materialised fine planes (bilinear_upsample + the stored-plane union select) against
      the virtual select;
per-kernel times (mask, one count pass, one step, apply), (a) against (b) bit for bit, algorithmic bytes per kernel
against the HBM copy bandwidth measured in the same run.  CUDA events, warmed up; card name and power limit first.
    python profiles/prof_fine.py [reps]"""
import ctypes
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hsr_b200 import _lib, kernels, synthetic  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("card:", smi[0] if smi else torch.cuda.get_device_name(dev))


def timed(fn, r=reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(r):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / r


src = torch.empty(1 << 30, dtype=torch.float32, device=dev)
dst = torch.empty_like(src)
hbm = 2 * src.numel() * 4 / timed(lambda: dst.copy_(src), 10) / 1e6
print(f"HBM copy bandwidth (measured, 4 GiB d2d): {hbm:.0f} GB/s")
del src, dst

Hr, Wr, B = 1280, 1242, 285
F = 6
w = synthetic.emit_wavelengths()
good = synthetic.good_band_mask(w)
raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, dev, good=good)
gx, gy = (torch.from_numpy(a).to(dev) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
src_gt = (-118.60, 0.000542232520256367, 0.0, 34.90, 0.0, -0.000542232520256367)
s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
target = hwarp.s2_target(src_gt, gx.shape, s2g)
Hd, Wd = target.shape
n10 = Hd * Wd * F * F
print(f"60 m target {Hd}x{Wd} -> 10 m {Hd * F}x{Wd * F} = {n10 / 1e6:.1f} Mpx per plane, factor {F}")

GB = 1e9


def report(name, ms, nbytes):
    print(f"  {name:<44s} {ms:8.3f} ms   {nbytes / GB:6.3f} GB  {nbytes / ms / 1e6:7.0f} GB/s  "
          f"{nbytes / ms / 1e6 / hbm:5.2f} of copy bw")


lib = _lib.lib()
for deg in (2, 4):
    for stretch in (None, (2, 98)):
        ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=deg, device=dev, stretch=stretch)
        K = ps.K
        x0 = ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((K, Hd, Wd), device=dev), target)
        s2 = synthetic.s2_reference_torch(torch.nan_to_num(x0.bands), seed=1)
        res = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target)
        coarse = K * Hd * Wd * 4
        plane10 = K * n10 * 4
        print(f"deg {deg}, stretch {stretch}, K = {K}  (60 m planes {coarse / 1e6:.0f} MB, 10 m planes {plane10 / GB:.2f} GB)")
        out_a = kernels.alloc_planes(K, (Hd * F, Wd * F), dev)

        def path_a():
            return ps.matched_fine(res, F, out=out_a)

        def path_b():
            x10 = kernels.bilinear_upsample(res.bands, F)
            m10 = kernels.fit_mask(x10, None, gate_k=-1)
            lim = kernels.masked_percentiles_union([(x10, m10)], stretch) if stretch is not None else None
            lo, hi = ps.clip
            _, out = kernels.poly_solve_apply(x10, res.moments, m10, deg, min_count=ps.min_count, lo=lo, hi=hi,
                                              x_stretch=lim)
            return out, m10, lim

        fa = path_a()
        ob, mb, lb = path_b()
        torch.cuda.synchronize()
        same = torch.equal(fa.matched.view(torch.int32), ob.view(torch.int32)) and torch.equal(fa.mask, mb)
        if stretch is not None:
            same = same and torch.equal(fa.x_limits.view(torch.int64), lb.view(torch.int64))
        print(f"  (a) == (b) bit for bit (planes, mask{', limits' if stretch else ''}): {same}")
        del ob, mb, lb
        ta, tb = [], []
        for _ in range(3):                                  # alternated
            ta.append(timed(path_a))
            tb.append(timed(lambda: path_b()))
        print(f"  (a) matched_fine        {' '.join(f'{t:7.3f}' for t in ta)} ms   min {min(ta):.3f}")
        print(f"  (b) chain of kernels    {' '.join(f'{t:7.3f}' for t in tb)} ms   min {min(tb):.3f}   "
              f"(b) / (a) = {min(tb) / min(ta):.2f}")
        # per kernel
        m10 = torch.empty((Hd * F, Wd * F), dtype=torch.bool, device=dev)
        report("fine mask (bilinear_fine_mask)", timed(lambda: kernels.bilinear_fine_mask(res.bands, F, out=m10)),
               coarse + n10)
        lim = fa.x_limits
        report("fused apply (bilinear_apply)",
               timed(lambda: kernels.bilinear_apply(res.bands, F, res.coeffs, x_stretch=lim, out=out_a, mask_out=m10)),
               coarse + plane10 + n10)
        if stretch is not None:
            q = torch.tensor([stretch[0] / 100, stretch[1] / 100], dtype=torch.float64, device=dev)
            st = torch.empty(lib.hsr_union_select_state_bytes(2, K) + 256, dtype=torch.uint8, device=dev)
            sp = st.data_ptr() + (-st.data_ptr()) % 256
            hist = torch.empty(lib.hsr_union_select_hist_doubles(2, K), dtype=torch.float64, device=dev)
            lout = torch.empty((K, 2), dtype=torch.float64, device=dev)
            sps = res.bands.stride(0)
            cs = torch.cuda.current_stream().cuda_stream
            more = ctypes.c_int(0)

            def virtual_select():
                return kernels.masked_percentiles_union([(res.bands, m10)], stretch, factor=F)

            def stored_select():
                x10 = kernels.bilinear_upsample(res.bands, F)
                return kernels.masked_percentiles_union([(x10, m10)], stretch)

            for p in range(4):
                lib.hsr_union_select_begin(q.data_ptr(), 2, K, sp, hist.data_ptr(), cs)
                for pp in range(p):                          # bring the state to pass p
                    lib.hsr_union_select_count_bilinear(res.bands.data_ptr(), sps, Hd, Wd, F, m10.data_ptr(), K, 2, pp,
                                                        sp, hist.data_ptr(), cs)
                    lib.hsr_union_select_step(2, K, pp, sp, hist.data_ptr(), lout.data_ptr(), ctypes.byref(more), cs)
                report(f"virtual count, pass {p}",
                       timed(lambda: lib.hsr_union_select_count_bilinear(res.bands.data_ptr(), sps, Hd, Wd, F,
                                                                         m10.data_ptr(), K, 2, p, sp, hist.data_ptr(),
                                                                         cs)),
                       coarse + n10)
            print(f"  {'union step (one pass)':<44s} "
                  f"{timed(lambda: lib.hsr_union_select_step(2, K, 0, sp, hist.data_ptr(), lout.data_ptr(), None, cs)):8.3f} ms")
            tv, ts = [], []
            for _ in range(3):
                tv.append(timed(virtual_select))
                ts.append(timed(stored_select))
            print(f"  (c) virtual select      {' '.join(f'{t:7.3f}' for t in tv)} ms   min {min(tv):.3f}   "
                  f"({(4 * (coarse + n10)) / GB:.3f} GB algorithmic)")
            print(f"  (c) upsample + stored select {' '.join(f'{t:7.3f}' for t in ts)} ms   min {min(ts):.3f}   "
                  f"({(coarse + plane10 + 4 * (plane10 + n10)) / GB:.3f} GB algorithmic)")
            x10 = kernels.bilinear_upsample(res.bands, F)
            report("bilinear_upsample (stored fine planes)", timed(lambda: kernels.bilinear_upsample(res.bands, F, out=x10)),
                   coarse + plane10)
            report("stored union select (4 counts + 4 steps)", timed(lambda: kernels.masked_percentiles_union([(x10, m10)], stretch)),
                   4 * (plane10 + n10))
            del x10
        print(f"  algorithmic bytes: (a) {(coarse + n10 + (4 * (coarse + n10) if stretch else 0) + coarse + plane10 + n10) / GB:.2f} GB, "
              f"(b) {(coarse + plane10 + plane10 + n10 + (4 * (plane10 + n10) if stretch else 0) + plane10 + n10 + plane10) / GB:.2f} GB")
        del out_a, fa, res, x0, s2
        torch.cuda.empty_cache()
