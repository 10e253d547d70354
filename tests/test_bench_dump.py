"""bench.py --dump-outputs: the arrays it writes, their sample and size, and the configs it refuses."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_samples_every_per_pixel_array_at_the_same_pixels(tmp_path):
    Ho, Wo, K = 1685, 1667, 12                                       # the granule config's ortho grid
    planes = torch.arange(K * Ho * (Wo + 13), dtype=torch.float32).view(K, Ho, Wo + 13)[:, :, :Wo]   # padded plane stride
    mask = torch.rand((Ho, Wo), generator=torch.Generator().manual_seed(0)) < 0.5
    coeffs = torch.randn((K, 1, 3), dtype=torch.float64)
    bench.dump_outputs(str(tmp_path), {"bands": planes, "valid": mask, "coeffs": coeffs}, (Ho, Wo))
    assert sorted(os.listdir(tmp_path)) == ["bands.npy", "coeffs.npy", "valid.npy"]
    idx = np.sort(np.random.default_rng(0).choice(Ho * Wo, size=bench.DUMP_SAMPLE_PX, replace=False))
    bands, valid, c = (np.load(tmp_path / f"{n}.npy") for n in ("bands", "valid", "coeffs"))
    assert bands.dtype == np.float32 and np.array_equal(bands, planes.reshape(K, -1)[:, idx].numpy())
    assert valid.dtype == np.float32 and np.array_equal(valid, mask.reshape(-1)[idx].numpy().astype(np.float32))
    assert c.dtype == np.float64 and np.array_equal(c, coeffs.numpy())
    # bands, matched (same size), valid, fit mask, coefficients: within 64 MB
    assert 2 * bands.nbytes + 2 * valid.nbytes + c.nbytes <= 64 * 2 ** 20


def test_dump_outputs_refused_where_it_is_not_implemented(tmp_path):
    for extra in (["--config", "tiles"], ["--impl", "reference"]):
        proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path)] + extra,
                              capture_output=True, text=True, timeout=120)
        assert proc.returncode == 2 and "--dump-outputs" in proc.stderr
