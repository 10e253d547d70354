"""The benchmark step (glt_stream<SRF>, poly_moments, moments_finalize, solve_apply) captured into a CUDA graph and
replayed, without the host's launch overhead.
    python profiles/prof_step_graph.py [reps]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hsr_b200 import kernels, synthetic  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 100
dev = torch.device("cuda", 0)
Hr, Wr, B = synthetic.GRANULE_RAW_SHAPE
w = synthetic.emit_wavelengths()
good = synthetic.good_band_mask(w)
ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device=dev)
gx_np, gy_np = synthetic.rotation_glt(Hr, Wr, 25.0)
gx, gy = torch.from_numpy(gx_np).to(dev), torch.from_numpy(gy_np).to(dev)
Ho, Wo = gx_np.shape
sets = []
for si in range(2):                                  # two input sets alternate, as in bench.py: nothing of step i is in L2 for step i + 1
    raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 1000 * si, dev, good)
    b0 = ps.bands_from_raw(raw, gx, gy)[0]
    s2 = kernels.alloc_planes(ps.K, (Ho, Wo), dev)
    s2.copy_(synthetic.s2_reference_torch(b0, seed=1 + si))
    sets.append((raw, s2))
bands = kernels.alloc_planes(ps.K, (Ho, Wo), dev)
matched = kernels.alloc_planes(ps.K, (Ho, Wo), dev)
graphs = []
for raw, s2 in sets:
    fn = lambda raw=raw, s2=s2: ps.synthesize(raw, gx, gy, s2, bands_out=bands, matched_out=matched)   # noqa: E731
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    graphs.append(g)
for i in range(10):
    graphs[i & 1].replay()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(reps):
    graphs[i & 1].replay()
e1.record()
torch.cuda.synchronize()
print(f"{e0.elapsed_time(e1) / reps:.4f} ms per step", flush=True)
