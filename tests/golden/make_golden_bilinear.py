"""Generate tests/golden/bilinear_up_seeded.npz: the output of hsr_bilinear_upsample_f32 on small seeded planes holding
NaN, +-Inf and the -9999 fill, at factors 1, 2, 3 and 6, with and without nodata.  Stored with its inputs, so that
tests/test_gpu_fine_grid.py can check that a later library (the interpolation moved into the shared
bilinear_up_value helper) gives the same bits.  Needs a GPU; the library is given on the command line, so the file can
be produced by the library of the commit before the change:

    python tests/golden/make_golden_bilinear.py path/to/libhsr_b200.so [out.npz]
"""
import ctypes
import os
import sys

import numpy as np
import torch

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "bilinear_up_seeded.npz")


def cases():
    rng = np.random.default_rng(20261021)
    for i, (C, Hs, Ws, factor, nodata) in enumerate(((3, 9, 11, 6, None), (2, 7, 5, 3, None), (1, 1, 1, 6, None),
                                                     (4, 12, 13, 2, None), (3, 6, 8, 1, None), (2, 9, 7, 6, -9999.0),
                                                     (5, 4, 15, 3, -9999.0), (1, 3, 2, 2, 0.5))):
        x = (rng.random((C, Hs, Ws)) * 2 - 0.5).astype(np.float32)
        flat = x.reshape(-1)
        n = flat.size
        for v, frac in ((np.nan, 0.05), (np.inf, 0.03), (-np.inf, 0.03), (-9999.0, 0.1), (0.5, 0.05), (-0.0, 0.03)):
            flat[rng.random(n) < frac] = v
        yield f"c{i}", x, factor, nodata


def main():
    lib = ctypes.CDLL(sys.argv[1])
    out = sys.argv[2] if len(sys.argv) > 2 else OUT
    fn = lib.hsr_bilinear_upsample_f32
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int,
                   ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    blob = {}
    for name, x, f, nd in cases():
        C, Hs, Ws = x.shape
        src = torch.from_numpy(x).cuda()
        dst = torch.empty((C, Hs * f, Ws * f), dtype=torch.float32, device="cuda")
        rc = fn(src.data_ptr(), C, Hs, Ws, Hs * Ws, f, int(nd is not None), 0.0 if nd is None else nd, dst.data_ptr(),
                Hs * f * Ws * f, torch.cuda.current_stream().cuda_stream)
        assert rc == 0, rc
        blob[f"{name}/src"] = x
        blob[f"{name}/factor"] = np.int64(f)
        blob[f"{name}/nodata"] = np.float64(np.nan if nd is None else nd)
        blob[f"{name}/out"] = dst.cpu().numpy()
    np.savez_compressed(out, **blob)
    print("wrote", out, len(blob) // 4, "cases")


if __name__ == "__main__":
    main()
