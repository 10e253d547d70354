"""The fused GLT + SRF kernel on a 25-degree granule, on an all-nodata grid (with and without the valid / fit masks) and on
an all-nodata grid of 64 rows (the fixed cost).
   python profiles/prof_invalid_knobs.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hsr_b200 import kernels, synthetic                     # noqa: E402
from hsr_b200.s2_emit.srf import srf_fold_weights, synthetic_s2_srf   # noqa: E402

dev = torch.device("cuda:0")
Hr, Wr, B = synthetic.GRANULE_RAW_SHAPE
w = synthetic.emit_wavelengths()
good = synthetic.good_band_mask(w)
raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, dev, good)
gx_np, gy_np = synthetic.rotation_glt(Hr, Wr, 25.0)
W, names, _, fo = srf_fold_weights(w, synthetic_s2_srf(), good)
Wt, fod = torch.from_numpy(W).to(dev), torch.from_numpy(fo).to(dev)
K = len(names)
gx = torch.from_numpy(gx_np).to(dev)
gy = torch.from_numpy(gy_np).to(dev)
out = kernels.alloc_planes(K, gx.shape, dev)
fm = torch.empty(gx.shape, dtype=torch.bool, device=dev)


def timed(f, reps=50):
    for _ in range(5):
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


z = torch.zeros_like(gx)
a = timed(lambda: kernels.glt_srf(raw, gx, gy, Wt, fod, bands_out=out, want_diag=False, fit_mask_out=fm, gate_k=0))
b = timed(lambda: kernels.glt_srf(raw, z, z, Wt, fod, bands_out=out, want_diag=False, fit_mask_out=fm, gate_k=0))
c = timed(lambda: kernels.glt_srf(raw, z, z, Wt, fod, bands_out=out, want_diag=False, want_valid=False))
small = z[:64].contiguous()
outs = kernels.alloc_planes(K, small.shape, dev)
d = timed(lambda: kernels.glt_srf(raw, small, small, Wt, fod, bands_out=outs, want_diag=False, want_valid=False))
print(f"granule {a:7.4f}   all-nodata {b:7.4f}   all-nodata, no valid / fit mask {c:7.4f}   64 rows only (fixed cost) {d:7.4f} ms", flush=True)
