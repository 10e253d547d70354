"""Host-side logic that needs no GPU: SRF weight folding, argument/error behaviour of the
reference-compatible wrappers, unit sharding, and the world_size-2 moment all-reduce on gloo."""
import os
import warnings

import numpy as np
import pytest
import torch

from hsr_b200 import dist as hdist
from hsr_b200 import kernels, synthetic
from hsr_b200.s2_emit import poly_regression, srf, synth
from oracle import srf as osrf

warnings.filterwarnings("ignore", category=RuntimeWarning)


def test_srf_fold_weights_equals_reference_integral():
    w = synthetic.emit_wavelengths()
    good = synthetic.good_band_mask(w)
    table = srf.synthetic_s2_srf()
    cube = synthetic.raw_cube_spectra_np((5, 4, 285), seed=3, good=good)
    cube[0, 0] = -9999.0
    for gm in (good, None):
        W, names, none_bands, fill_out = srf.srf_fold_weights(w, table, gm)
        ref = osrf.pseudo_s2_srf_integral(cube, w, table, gm)
        assert [b for b in table if ref[b] is None] == none_bands
        assert names == [b for b in table if ref[b] is not None]
        assert W.dtype == np.float32 and W.shape == (285, len(names))
        got = cube.astype(np.float64) @ W.astype(np.float64)
        for i, b in enumerate(names):
            np.testing.assert_allclose(got[..., i], ref[b], rtol=2e-6, atol=1e-9)
        np.testing.assert_allclose(fill_out, -9999.0, rtol=1e-6)
    W, names, none_bands, _ = srf.srf_fold_weights(w, table, good)
    assert none_bands == ["B10"] and len(names) == 12
    # each folded response is one contiguous run of bands (what the kernel's run table relies on for speed)
    for i in range(W.shape[1]):
        nz = np.flatnonzero(W[:, i])
        assert nz.size > 0


def test_trapezoid_weights_regroup_np_trapz():
    rng = np.random.default_rng(0)
    x = np.sort(rng.uniform(400, 2500, size=37))
    y = rng.normal(size=37)
    trapz = getattr(np, "trapezoid", None) or np.trapz
    assert abs(float(np.sum(srf.trapezoid_weights(x) * y)) - float(trapz(y, x=x))) < 1e-9


def test_synthetic_srf_has_reference_format():
    table = srf.synthetic_s2_srf()
    assert list(table) == srf.S2_BANDS_13
    for lam, rsp in table.values():
        assert lam.dtype == np.float64 and rsp.dtype == np.float64
        assert np.all(np.diff(lam) > 0) and np.all(rsp > 0) and np.all(np.isfinite(rsp))


def test_rotation_glt_matches_survey_numbers():
    gx, gy = synthetic.rotation_glt(1280, 1242, 25.0)
    assert gx.shape == (1685, 1667) and gx.dtype == np.int32
    valid = (gx != 0) & (gy != 0)
    assert abs(valid.mean() - 0.566) < 0.002
    assert gx.max() <= 1242 and gy.max() <= 1280 and gx.min() >= 0


def test_kernels_refuse_cpu_tensors():
    raw = torch.zeros(4, 4, 8)
    g = torch.ones(4, 4, dtype=torch.int32)
    with pytest.raises(TypeError, match="no CPU path"):
        kernels.glt_ortho(raw, g, g)
    with pytest.raises(TypeError):
        kernels.srf_integrate(raw, torch.zeros(8, 2))
    with pytest.raises(TypeError):
        kernels.poly_fit(torch.zeros(2, 16), torch.zeros(2, 16), None, 2)
    with pytest.raises(TypeError):
        kernels.glt_ortho(np.zeros((4, 4, 8), np.float32), g, g)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU error path")
def test_wrappers_fail_loudly_without_a_gpu():
    w = synthetic.emit_wavelengths()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        synth.pseudo_s2_srf_integral(np.zeros((2, 2, 285), np.float32), w, srf.synthetic_s2_srf())
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        poly_regression.apply_poly_rgb(np.zeros((2, 2, 3), np.float32), np.zeros((3, 3)))


def test_wrapper_argument_errors_match_reference():
    w = synthetic.emit_wavelengths()
    table = srf.synthetic_s2_srf()
    with pytest.raises(ValueError, match=r"R must be \(H,W,B\)"):
        synth.pseudo_s2_srf_integral(np.zeros((2, 285), np.float32), w, table)
    with pytest.raises(ValueError, match="emit_w must be"):
        synth.pseudo_s2_srf_integral(np.zeros((2, 2, 285), np.float32), w[:-1], table)
    with pytest.raises(ValueError, match="None/missing"):
        synth.pseudo_s2_rgb({"B4": None, "B3": np.zeros((2, 2)), "B2": np.zeros((2, 2))})
    with pytest.raises(ValueError, match="targets must be"):
        poly_regression.fit_ot_poly_rgb(np.zeros((4, 4, 3)), np.zeros((4, 4, 3)), np.ones((4, 4), bool), targets="x")


def test_shard_units_and_rows():
    for n, ws in ((64, 8), (7, 4), (3, 8), (0, 2)):
        seen = []
        for r in range(ws):
            mine = hdist.shard_units(n, r, ws)
            seen += mine
            assert len(mine) in (n // ws, n // ws + 1)
        assert sorted(seen) == list(range(n))
    spans = [hdist.shard_rows(8192, r, 8) for r in range(8)]
    assert spans[0] == (0, 1024) and spans[-1] == (7168, 8192)
    spans = [hdist.shard_rows(1685, r, 4, align=32) for r in range(4)]
    assert spans[0][0] == 0 and spans[-1][1] == 1685
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    with pytest.raises(ValueError):
        hdist.shard_units(4, 2, 2)


def _moments_np(x, y, deg):
    pw = np.vander(x.astype(np.float64), 2 * deg + 1, increasing=True)
    S = pw.sum(0)
    T = (pw[:, : deg + 1] * y.astype(np.float64)[:, None]).sum(0)
    return np.concatenate([S, T])


def _gloo_worker(rank, world_size, port, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size),
                      LOCAL_RANK=str(rank))
    r, ws, dev = hdist.init_from_env(backend="gloo")
    assert (r, ws) == (rank, world_size) and hdist.world() == (rank, world_size)
    rng = np.random.default_rng(5)
    units = [(rng.uniform(0.05, 0.8, 500).astype(np.float32), None) for _ in range(5)]
    units = [(x, (-0.3 * x.astype(np.float64) ** 2 + 1.1 * x + 0.02).astype(np.float32)) for x, _ in units]
    mine = hdist.shard_units(len(units), rank, world_size)
    per_unit = [torch.from_numpy(_moments_np(*units[i], 2))[None] for i in mine]
    mom = hdist.sum_moments(per_unit)
    hdist.allreduce_moments(mom)
    np.save(os.path.join(tmpdir, f"mom_{rank}.npy"), mom.numpy())
    torch.distributed.destroy_process_group()


def test_min_norm_from_moments_equals_np_polyfit_on_rank_deficient_series():
    """Host repair of rank-deficient fits (np.polyfit returns the SVD minimum-norm solution, the device's Gauss-Jordan
    solve NaN): from the normal-equation moments alone, for constant / two-valued / three-valued x and a full-rank one."""
    import warnings

    from hsr_b200._host import min_norm_from_moments, repair_rank_deficient
    rng = np.random.default_rng(0)

    def moments(x, y, deg):
        return np.array([np.sum(x ** j) for j in range(2 * deg + 1)] + [np.sum(x ** j * y) for j in range(deg + 1)])

    rows, refs = [], []
    for x, deg, rank in ((np.full(500, 0.37), 2, 1), (rng.choice([0.2, 0.7], 500), 3, 2), (rng.choice([0.1, 0.5, 0.9], 800), 4, 3),
                         (rng.random(500), 2, 3)):
        y = rng.random(x.size)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = np.polyfit(x, y, deg)
        c, r = min_norm_from_moments(moments(x, y, deg), deg)
        assert r == rank and np.abs(c - ref).max() <= 1e-10 * np.abs(ref).max()
        if deg == 2:
            rows.append(moments(x, y, deg)), refs.append(ref)
    bad = np.full((2, 3), np.nan)
    bad[1] = refs[1]                                               # the full-rank row keeps the device's coefficients
    with pytest.warns(np.exceptions.RankWarning):
        fixed = repair_rank_deficient(bad, np.stack(rows), 2)
    assert np.allclose(fixed[0], refs[0], rtol=1e-10) and np.array_equal(fixed[1], refs[1])
    few = repair_rank_deficient(np.array([[0.0, 1.0, 0.0]]), rows[0][None], 2, min_count=1000)   # below min_count: untouched
    assert np.array_equal(few, [[0.0, 1.0, 0.0]])


def test_shard_rows_balanced_by_weights():
    """Row slabs balanced by work (bench --config mosaic): contiguous, aligned, covering, and within one aligned step
    of equal cumulative weight."""
    n = 1000
    w = np.concatenate([np.linspace(0, 10, 500), np.linspace(10, 0, 500)])          # a rotated swath: busy in the middle
    for world in (1, 2, 3, 8):
        slabs = [hdist.shard_rows(n, r, world, align=8, weights=w) for r in range(world)]
        assert slabs[0][0] == 0 and slabs[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(slabs, slabs[1:]))
        assert all(a % 8 == 0 for a, _ in slabs)
        work = [w[a:b].sum() for a, b in slabs]
        assert max(work) <= w.sum() / world + 8 * w.max() + 1e-9
    even = [hdist.shard_rows(n, r, 8, align=8) for r in range(8)]
    assert max(w[a:b].sum() for a, b in even) > 1.5 * w.sum() / 8                    # what balancing buys
    assert hdist.shard_rows(n, 2, 4, weights=np.zeros(n)) == hdist.shard_rows(n, 2, 4)
    with pytest.raises(ValueError):
        hdist.shard_rows(n, 0, 2, weights=w[:10])


def test_moment_allreduce_world_size_2_gloo(tmp_path, monkeypatch):
    import torch.multiprocessing as mp

    # the workers are CPU ranks: with a GPU visible, init_from_env would bind rank 1 to cuda:1, absent on a one-GPU box
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    port = 29500 + (os.getpid() % 400)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    m0 = np.load(tmp_path / "mom_0.npy")
    m1 = np.load(tmp_path / "mom_1.npy")
    assert np.array_equal(m0, m1)
    rng = np.random.default_rng(5)
    xs = [rng.uniform(0.05, 0.8, 500).astype(np.float32) for _ in range(5)]
    ys = [(-0.3 * x.astype(np.float64) ** 2 + 1.1 * x + 0.02).astype(np.float32) for x in xs]
    allx, ally = np.concatenate(xs), np.concatenate(ys)
    np.testing.assert_allclose(m0[0], _moments_np(allx, ally, 2), rtol=1e-12)
    # the all-reduced normal equations give the global fit
    S, T = m0[0][:5], m0[0][5:]
    G = np.array([[S[i + j] for j in range(3)] for i in range(3)])
    c = np.linalg.solve(G, T)[::-1]
    np.testing.assert_allclose(c, np.polyfit(allx.astype(np.float64), ally.astype(np.float64), 2), rtol=1e-6)


def test_allreduce_is_identity_for_single_process():
    m = torch.arange(8, dtype=torch.float64).view(1, 8)
    assert hdist.allreduce_moments(m.clone()).equal(m)
    with pytest.raises(TypeError):
        hdist.allreduce_moments(torch.zeros(2, 8))


def test_gdal_export_helpers_build_the_reference_commands(monkeypatch, tmp_path):
    """The GDAL-facing helpers of emit_proj.py (:248-306, :399-560) keep their names, signatures and command lines;
    no GDAL here, so run_cmd is intercepted."""
    from hsr_b200.EMIT_data import emit_proj, gdal_export
    calls = []
    monkeypatch.setattr(gdal_export, "run_cmd", lambda cmd, check=True: calls.append(list(cmd)) or {"cmd": list(cmd)})
    monkeypatch.setattr(gdal_export.shutil, "which", lambda c: "/usr/bin/gdal_edit.py" if c == "gdal_edit.py" else None)
    rec = emit_proj.export_uint16_deflate_geotiff("a.bin", "a.tif", assign_epsg="EPSG:4326", scale_mode="emit_reflectance_0_1")
    cmd = rec["cmd"]
    assert cmd[:5] == ["gdal_translate", "-of", "GTiff", "-ot", "UInt16"] and cmd[-2:] == ["a.bin", "a.tif"]
    assert " ".join(cmd).count("-scale 0 1 0 10000") == 1 and "-a_nodata 65535" in " ".join(cmd) and "ZLEVEL=1" in " ".join(cmd)
    assert cmd[cmd.index("-a_srs") + 1] == "EPSG:4326" and "scale_factor=0.0001" in cmd
    plain = emit_proj.export_uint16_deflate_geotiff("a.bin", "b.tif", zlevel=6)["cmd"]
    assert "-scale" not in plain and "-a_srs" not in plain and "ZLEVEL=6" in " ".join(plain)
    calls.clear()
    rec = emit_proj.export_loc_uint16_deflate_geotiff("loc.bin", "loc.tif", elev_range=(0.0, 6553.5))
    line = " ".join(calls[0])
    assert "-scale_1 -180.0 180.0 0 65535 -exponent_1 1" in line and "-scale_3 0.0 6553.5 0 65535 -exponent_3 1" in line
    assert calls[1][0] == "gdal_edit.py" and calls[1][-1] == "loc.tif" and "-offset" in calls[1]     # decode metadata written
    d = rec["uint16_decode"]
    assert d["offsets"] == [-180.0, -90.0, 0.0] and abs(d["scales"][2] - 0.1) < 1e-12 and d["nodata_uint16"] == 0
    assert d["ranges"][1] == [-90.0, 90.0] and "raw*scale + offset" in d["note"]
    assert emit_proj.raster_meta(str(tmp_path / "missing.tif")) == {"path": str(tmp_path / "missing.tif"), "exists": False}
    # the range rule of _sample_band_minmax (:478-493)
    a = np.array([[0.0, 1.0, 2.0, np.nan], [-9999.0, 3.0, 4.0, np.inf]], np.float32)
    lo, hi = gdal_export._robust_range(a, -9999.0, 0.0, 100.0)
    assert (lo, hi) == (0.0, 4.0)
    assert gdal_export._robust_range(np.full((3, 3), -9999.0, np.float32), -9999.0, 1, 99) == (0.0, 1.0)
    assert gdal_export._robust_range(np.full((3, 3), 7.0, np.float32), -9999.0, 1, 99) == (7.0, 8.0)
    with pytest.raises(ImportError):
        emit_proj.export_obs_uint16_deflate_geotiff("obs.bin", "obs.tif", nodata_float=-9999.0)     # needs rasterio
    assert emit_proj._compute_te is not None and emit_proj._intersect((0, 0, 2, 2), (1, 1, 3, 3)) == (1, 1, 2, 2)


def test_envi_reader_round_trips_every_interleave(tmp_path):
    """load_emit_envi_rfl (s2_emit/emit_io.py:7-16): (lines, samples, bands) whatever the interleave / type / byte order,
    multi-line brace lists in the header."""
    from hsr_b200.s2_emit import emit_io, load_emit_envi_rfl
    rng = np.random.default_rng(0)
    H, W, B = 5, 7, 4
    cube = rng.random((H, W, B)).astype(np.float32)
    layouts = {"bil": cube.transpose(0, 2, 1), "bip": cube, "bsq": cube.transpose(2, 0, 1)}
    for inter, arr in layouts.items():
        for code, dt, order in ((4, "<f4", 0), (4, ">f4", 1), (5, "<f8", 0), (12, "<u2", 0)):
            data = (arr * 1000).astype(dt) if code == 12 else arr.astype(dt)
            p = tmp_path / f"c_{inter}_{code}_{order}"
            with open(p, "wb") as fh:
                fh.write(b"x" * 16)
                fh.write(np.ascontiguousarray(data).tobytes())
            (tmp_path / f"c_{inter}_{code}_{order}.hdr").write_text(
                "ENVI\ndescription = {\n  a cube,\n  two lines }\n"
                f"samples = {W}\nlines   = {H}\nbands = {B}\nheader offset = 16\ndata type = {code}\n"
                f"interleave = {inter}\nbyte order = {order}\n" "wavelength = { 400.0 , 500.0 ,\n 600.0 , 700.0 }\n")
            R = load_emit_envi_rfl(str(p) + ".hdr", str(p))
            want = (cube * 1000).astype("u2").astype(np.float32) if code == 12 else cube.astype(dt).astype(np.float32)
            assert R.shape == (H, W, B) and R.dtype == np.float32 and np.array_equal(R, want), (inter, code, order)
            raw = load_emit_envi_rfl(str(p) + ".hdr", str(p), as_float32=False)
            assert raw.dtype == np.dtype(dt).newbyteorder("=") and raw.dtype.isnative
    h = emit_io.read_envi_header(tmp_path / "c_bil_4_0.hdr")
    assert h["description"] == "a cube, two lines" and np.array_equal(emit_io.envi_list(h["wavelength"]), [400, 500, 600, 700])
    (tmp_path / "bad.hdr").write_text("samples = 3\n")
    with pytest.raises(ValueError):
        load_emit_envi_rfl(str(tmp_path / "bad.hdr"), str(tmp_path / "c_bil_4_0"))
    with pytest.raises(ImportError):
        emit_io.load_emit_wavelengths_from_nc(str(tmp_path / "none.nc"))            # no HDF5 reader in this image


def test_load_s2_srf_from_xlsx_format_with_a_fake_workbook(monkeypatch):
    """load_s2_srf_from_xlsx / pick_sheet_name (s2_emit/srf.py:13-52): sheet choice, column naming, the finite & > 0 row
    filter, KeyError for a missing band column — on a fake workbook (no openpyxl / network here)."""
    import pandas as pd
    lam = np.arange(300.0, 310.0)
    frame = pd.DataFrame({"SR_WL": list(lam[:-1]) + ["n/a"],
                          "S2A_SR_AV_B2": [0.0, 0.1, 0.2, np.nan, 0.4, -0.1, 0.6, 0.7, 0.8, 0.9],
                          "S2A_SR_AV_B3": np.linspace(0.0, 0.9, 10)})

    class FakeBook:
        sheet_names = ["Readme", "Spectral Responses (S2A)", "Spectral Responses (S2B)"]

        def __init__(self, url):
            self.url = url

        def parse(self, sheet):
            assert sheet == "Spectral Responses (S2A)"
            return frame

    monkeypatch.setattr(pd, "ExcelFile", FakeBook)
    out = srf.load_s2_srf_from_xlsx("fake.xlsx", bands=["B2", "B3"])
    assert list(out) == ["B2", "B3"]
    assert np.array_equal(out["B2"][0], [301, 302, 304, 306, 307, 308]) and np.allclose(out["B2"][1], [0.1, 0.2, 0.4, 0.6, 0.7, 0.8])
    assert out["B3"][0][0] == 301 and out["B3"][0][-1] == 308 and out["B3"][1].dtype == np.float64   # 0 response and 'n/a' row dropped
    assert srf.pick_sheet_name(FakeBook("x"), "s2b") == "Spectral Responses (S2B)"
    with pytest.raises(ValueError):
        srf.pick_sheet_name(FakeBook("x"), "S2C")
    with pytest.raises(KeyError):
        srf.load_s2_srf_from_xlsx("fake.xlsx", bands=["B2", "B8A"])
    # and the reference's synth.py accepts the dict unchanged through our wrapper
    w = synthetic.emit_wavelengths()
    R = np.random.default_rng(0).random((3, 4, w.size)).astype(np.float32)
    tab = {"B2": (np.arange(440.0, 540.0), np.ones(100)), "B10": (np.arange(1360.0, 1390.0), np.ones(30))}
    Wf, names, none_bands, _ = srf.srf_fold_weights(w, tab, synthetic.good_band_mask(w))
    assert names == ["B2"] and none_bands == ["B10"] and Wf.shape == (w.size, 1)


def test_envi_writer_and_readers_agree(tmp_path):
    """What nc_to_envi writes (band-interleaved-by-line float32 + header) is what read_envi_bil and the
    load_emit_envi_rfl mirror read back, header lists included."""
    from hsr_b200.EMIT_data import nc_export
    from hsr_b200.s2_emit import emit_io
    rng = np.random.default_rng(4)
    cube = torch.from_numpy(rng.random((9, 13, 5)).astype(np.float32))
    cube[2, 3, 1] = float("nan")
    p = nc_export.write_envi_bil(tmp_path / "cube", cube, {"data ignore value": -9999.0, "wavelength": [400.0, 450.5, 500.0, 550.0, 600.25],
                                                          "map info": ["UTM", 1, 1, 300000.0, 3900000.0, 60.0, 60.0, 11, "North", "WGS-84"]},
                                 rows_per_chunk=4)
    back, hdr = nc_export.read_envi_bil(p)
    assert back.shape == (9, 13, 5) and np.array_equal(back, cube.numpy(), equal_nan=True)
    assert hdr["interleave"] == "bil" and hdr["data ignore value"] == "-9999.0"
    R = emit_io.load_emit_envi_rfl(str(p) + ".hdr", str(p))
    assert np.array_equal(R, cube.numpy(), equal_nan=True)
    h = emit_io.read_envi_header(str(p) + ".hdr")
    assert np.array_equal(emit_io.envi_list(h["wavelength"]), [400.0, 450.5, 500.0, 550.0, 600.25]) and h["map info"].startswith("UTM , 1 , 1")
    # separate header path, as the UTM products use (<tag>.bin + <tag>.hdr)
    nc_export.write_envi_bil(tmp_path / "x.bin", cube, {}, hdr_path=tmp_path / "x.hdr")
    assert (tmp_path / "x.hdr").exists() and not (tmp_path / "x.bin.hdr").exists()
    assert np.array_equal(emit_io.load_emit_envi_rfl(str(tmp_path / "x.hdr"), str(tmp_path / "x.bin")), cube.numpy(), equal_nan=True)
