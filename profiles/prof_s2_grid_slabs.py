"""Timing of row bands on the Sentinel-2 grid (PairSynthesizer.synthesize_slab_on_s2_grid).

1. The granule workload of profiles/prof_s2_grid.py (raw 1280 x 1242 x 285, 25 degree GLT, the zone 11 60 m target
   1215 x 959, raw on the device) as 1, 2, 4 and 8 sequential bands against one synthesize_on_s2_grid call: the time
   of all bands and the halo, the ortho rows staged beyond the ortho rows one band over the whole target reads.
2. A mosaic onto a zone 11 60 m target (the configs[4] construction: raw mosaic in pinned host memory, 25 degree GLT,
   EMIT-like 0.000542 degree ortho pixels), dealt to N = 1, 2, 4, 8 ranks by dist.shard_rows.  With one process the
   bands of the N ranks run one after another on one GPU, each timed on its own: the largest is the time a rank of N
   would take with no contention and no exchange, which is not an N-GPU measurement.  Under torchrun (one process per
   GPU) every rank runs its band at once with a global fit over the peer exchange, and the step time is the maximum
   over the ranks.
CUDA events, warmed up; card name and power limit printed first.
    python profiles/prof_s2_grid_slabs.py [reps]
    torchrun --nproc-per-node=N profiles/prof_s2_grid_slabs.py [reps]"""
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hsr_b200 import dist as hdist  # noqa: E402
from hsr_b200 import synthetic  # noqa: E402
from hsr_b200.EMIT_data import warp as hwarp  # noqa: E402
from hsr_b200.pipeline import PairSynthesizer  # noqa: E402
from hsr_b200.s2_emit.srf import synthetic_s2_srf  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
rank, world, dev = hdist.init_from_env()
if rank == 0:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print("card:", smi[0] if smi else torch.cuda.get_device_name(dev), f"(x{torch.cuda.device_count()} visible)")
PIX = 0.000542232520256367


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


def bands_of(Hd, n):
    return [hdist.shard_rows(Hd, i, n) for i in range(n)]


w = synthetic.emit_wavelengths()
good = synthetic.good_band_mask(w)
ps = PairSynthesizer(w, synthetic_s2_srf(), good, deg=2, device=dev)

# ---------------------------------------------------------------------------------------------- 1. the granule
if world == 1:
    Hr, Wr, B = 1280, 1242, 285
    raw = synthetic.raw_cube_spectra_torch((Hr, Wr, B), 0, dev, good=good)
    gx, gy = (torch.from_numpy(a).to(dev) for a in synthetic.rotation_glt(Hr, Wr, 25.0))
    src_gt = (-118.60, PIX, 0.0, 34.90, 0.0, -PIX)
    s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=10980, height=10980)
    target = hwarp.s2_target(src_gt, gx.shape, s2g)
    Hd, Wd = target.shape
    s2 = synthetic.s2_reference_torch(torch.nan_to_num(
        ps.synthesize_on_s2_grid(raw, gx, gy, torch.zeros((ps.K, Hd, Wd), device=dev), target).bands), seed=1)
    one = ps.synthesize_on_s2_grid(raw, gx, gy, s2, target)
    o_one = None                      # ortho rows the whole target reads (one band)
    t_one = timed(lambda: ps.synthesize_on_s2_grid(raw, gx, gy, s2, target))
    print(f"granule: ortho {gx.shape[0]}x{gx.shape[1]} -> utm {Hd}x{Wd}; one synthesize_on_s2_grid call "
          f"{t_one:.3f} ms (cached coordinates)")
    s2b = {}
    for n in (1, 2, 4, 8):
        bands = bands_of(Hd, n)
        for t0, t1 in bands:
            s2b[(t0, t1)] = s2[:, t0:t1].contiguous()

        def run(bands=bands):
            return [ps.synthesize_slab_on_s2_grid(raw, gx, gy, s2b[b], target, b) for b in bands]

        res = run()
        torch.cuda.synchronize()
        staged = sum(r.ortho_rows[1] - r.ortho_rows[0] for r in res)
        o_one = o_one or staged
        stitched = torch.cat([r.bands for r in res], dim=1)
        same = torch.equal(stitched.view(torch.int32), one.bands.contiguous().view(torch.int32))
        t = timed(run)
        print(f"  {n} bands: {t:8.3f} ms for all ({t - t_one:+.3f} ms vs one call), ortho rows staged {staged} "
              f"(halo {staged - o_one:+d} rows over {o_one}), raw rows staged "
              f"{sum(r.raw_rows[1] - r.raw_rows[0] for r in res)}, bit-identical to one call: {same}")
    del raw, s2, one, s2b

# ---------------------------------------------------------------------------------------------- 2. the mosaic
Hr, Wr, B = 2400, 1242, 285                        # raw mosaic of ~2 granules along track, in pinned host memory
raw_np = synthetic.raw_cube_spectra_np((Hr, Wr, B), seed=7, good=good)
raw_host = torch.from_numpy(raw_np).pin_memory()
del raw_np
gxn, gyn = synthetic.rotation_glt(Hr, Wr, 25.0)
gx, gy = torch.from_numpy(gxn).to(dev), torch.from_numpy(gyn).to(dev)
src_gt = (-118.60, PIX, 0.0, 34.90, 0.0, -PIX)
# a zone 11 grid on the S2 lattice that holds the whole mosaic (one S2 tile is 109.8 km, the mosaic ~160 km)
s2g = hwarp.S2Grid(epsg=32611, x0=300000.0, y0=3900000.0, dx=10.0, dy=10.0, width=30000, height=30000)
target = hwarp.s2_target(src_gt, gx.shape, s2g)
Hd, Wd = target.shape
s2 = torch.rand((ps.K, Hd, Wd), device=dev) * 0.5 + 0.1
stage = torch.empty(Hr * Wr * B, dtype=torch.float32, device=dev)
if rank == 0:
    print(f"mosaic: raw {Hr}x{Wr}x{B} in pinned host memory, ortho {gx.shape[0]}x{gx.shape[1]} -> utm {Hd}x{Wd}")
if world == 1:
    base = None
    for n in (1, 2, 4, 8):
        times, rows = [], []
        for b in bands_of(Hd, n):
            s2s = s2[:, b[0]:b[1]].contiguous()
            times.append(timed(lambda b=b, s2s=s2s: ps.synthesize_slab_on_s2_grid(raw_host, gx, gy, s2s, target, b,
                                                                                    stage=stage)))
            r = ps.synthesize_slab_on_s2_grid(raw_host, gx, gy, s2s, target, b, stage=stage)
            rows.append(r.raw_rows[1] - r.raw_rows[0])
        base = base or max(times)
        print(f"  N={n} (sequential on one GPU): band time max {max(times):8.3f} ms, sum {sum(times):8.3f} ms, "
              f"speed-up of the max band over N=1 {base / max(times):.2f}x, raw rows staged per band max "
              f"{max(rows)} of {Hr}")
else:
    px = hdist.PeerExchange(device=dev, timeout_ms=20000)
    b = hdist.shard_rows(Hd, rank, world)
    s2s = s2[:, b[0]:b[1]].contiguous()

    def step():
        return ps.synthesize_slab_on_s2_grid(raw_host, gx, gy, s2s, target, b, stage=stage, exchange=px)

    t = timed(step)
    r = step()
    torch.cuda.synchronize()
    px.check()
    out = [None] * world
    dist.all_gather_object(out, (t, r.raw_rows[1] - r.raw_rows[0]))
    if rank == 0:
        ts = [o[0] for o in out]
        print(f"  N={world} ranks, global fit over the peer exchange: step time max over ranks {max(ts):8.3f} ms "
              f"(per rank {', '.join(f'{x:.3f}' for x in ts)}), raw rows staged per rank max "
              f"{max(o[1] for o in out)} of {Hr}")
    dist.barrier()
    px.close()
    dist.destroy_process_group()
