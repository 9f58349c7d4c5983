"""GPU: the file-level API and the CLI -- the reference's tests/test_flow_direction.py:121-160 with the
built-in GeoTIFF I/O standing in for GDAL's /vsimem, plus the added flow-accumulation driver."""
import threading
import time

import click.testing
import numpy as np
import pytest

import oracle
from oracle import synth
from conftest import load_golden
from overflow.constants import FLOW_DIRECTION_NODATA, FLOW_ACCUMULATION_NODATA
from overflow.flow_accumulation import flow_accumulation
from overflow.flow_direction import flow_direction
from overflow_b200.util.raster import create_raster, open_raster
from overflow_cli import flow_accumulation_cli, flow_direction_cli

pytestmark = pytest.mark.gpu


@pytest.fixture
def raster_file_path(tmp_path):
    """5x5 DEM of the reference's fixture (tests/test_flow_direction.py:21-50), nodata 0."""
    path = str(tmp_path / "test_raster_FDIR.tif")
    ds = create_raster(path, 5, 5, "Float32")
    band = ds.GetRasterBand(1)
    band.WriteArray(load_golden("kat.npz")["dir_dem"][1:-1, 1:-1])
    band.SetNoDataValue(0)
    ds.FlushCache()
    return path


def test_flow_direction_from_file(raster_file_path, tmp_path):
    out = str(tmp_path / "fdr.tif")
    flow_direction(raster_file_path, out, chunk_size=5)
    band = open_raster(out).GetRasterBand(1)
    assert band.GetNoDataValue() == FLOW_DIRECTION_NODATA
    assert np.array_equal(band.ReadAsArray(), load_golden("kat.npz")["dir_expected"])


def test_flow_direction_cli(raster_file_path, tmp_path):
    out = str(tmp_path / "fdr_cli.tif")
    result = click.testing.CliRunner().invoke(
        flow_direction_cli, ["--input_file", raster_file_path, "--output_file", out, "--chunk_size", "5"])
    assert result.exit_code == 0
    assert np.array_equal(open_raster(out).GetRasterBand(1).ReadAsArray(), load_golden("kat.npz")["dir_expected"])


def test_cli_failure_exits_non_zero(tmp_path):
    result = click.testing.CliRunner().invoke(
        flow_direction_cli, ["--input_file", str(tmp_path / "missing.tif"), "--output_file", str(tmp_path / "o.tif")])
    assert result.exit_code == 1
    assert "flow_direction failed with the following exception" in result.output


@pytest.mark.parametrize("chunk_size", [16, 50, 64, 4000])
def test_file_pipeline_is_chunk_size_invariant(tmp_path, chunk_size):
    dem = synth.punch_holes(synth.fractal(137, 211, beta=2.0, seed=5), frac=0.03, seed=6)
    src = str(tmp_path / "dem.tif")
    ds = create_raster(src, dem.shape[1], dem.shape[0], "Float32", geotransform=(0.0, 30.0, 0.0, 0.0, 0.0, -30.0))
    ds.GetRasterBand(1).WriteArray(dem)
    ds.GetRasterBand(1).SetNoDataValue(synth.NODATA)
    ds.FlushCache()
    fdr_path, fac_path = str(tmp_path / "fdr.tif"), str(tmp_path / "fac.tif")
    flow_direction(src, fdr_path, chunk_size=chunk_size)
    want_fdr = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1]
    fdr = open_raster(fdr_path).GetRasterBand(1).ReadAsArray()
    assert np.array_equal(fdr, want_fdr)
    result = click.testing.CliRunner().invoke(
        flow_accumulation_cli, ["--input_file", fdr_path, "--output_file", fac_path, "--chunk_size", str(chunk_size)])
    assert result.exit_code == 0, result.output
    out = open_raster(fac_path)
    band = out.GetRasterBand(1)
    assert band.GetNoDataValue() == FLOW_ACCUMULATION_NODATA
    assert out.GetGeoTransform() == pytest.approx((0.0, 30.0, 0.0, 0.0, 0.0, -30.0))
    assert np.array_equal(band.ReadAsArray(), oracle.flow_accumulation(want_fdr))


def test_flow_routing_files_equal_the_two_step_outputs(tmp_path):
    """DEM file -> both rasters in one pass: same bytes as flow_direction() then flow_accumulation()."""
    from overflow_cli import flow_routing_cli

    dem = synth.punch_holes(synth.fractal(150, 97, beta=2.5, seed=8), frac=0.03, seed=9)
    src = str(tmp_path / "dem.tif")
    ds = create_raster(src, dem.shape[1], dem.shape[0], "Float32", geotransform=(10.0, 30.0, 0.0, 20.0, 0.0, -30.0))
    ds.GetRasterBand(1).WriteArray(dem)
    ds.GetRasterBand(1).SetNoDataValue(synth.NODATA)
    ds.FlushCache()
    a_fdr, a_fac = str(tmp_path / "a_fdr.tif"), str(tmp_path / "a_fac.tif")
    b_fdr, b_fac = str(tmp_path / "b_fdr.tif"), str(tmp_path / "b_fac.tif")
    flow_direction(src, a_fdr, chunk_size=40)
    flow_accumulation(a_fdr, a_fac, chunk_size=40)
    result = click.testing.CliRunner().invoke(
        flow_routing_cli, ["--input_file", src, "--flow_direction_file", b_fdr, "--flow_accumulation_file", b_fac,
                           "--chunk_size", "64"])
    assert result.exit_code == 0, result.output
    for a, b in ((a_fdr, b_fdr), (a_fac, b_fac)):
        ra, rb = open_raster(a), open_raster(b)
        assert np.array_equal(ra.GetRasterBand(1).ReadAsArray(), rb.GetRasterBand(1).ReadAsArray())
        assert ra.GetRasterBand(1).GetNoDataValue() == rb.GetRasterBand(1).GetNoDataValue()
        assert ra.GetGeoTransform() == pytest.approx(rb.GetGeoTransform())
    want_fdr = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1]
    assert np.array_equal(open_raster(b_fac).GetRasterBand(1).ReadAsArray(), oracle.flow_accumulation(want_fdr))


# ---- the band pipeline of streaming.py (SURVEY 8f rank 1): the oracle's codes and counts, and those of the whole-raster
# host call (what the file drivers computed before Float32 DEMs streamed), for any band height
@pytest.mark.parametrize("band_rows", [1, 7, 64, 100, 5000])
def test_streamed_routing_equals_oracle_and_whole_raster(tmp_path, band_rows, monkeypatch):
    import torch

    from overflow_b200 import device as dev
    from overflow_b200.flow_routing import flow_routing_for_raster
    from overflow_b200.streaming import stream_routing

    dem = synth.punch_holes(synth.fractal(333, 257, beta=2.0, seed=15), frac=0.03, seed=16)
    src = str(tmp_path / "dem.tif")
    ds = create_raster(src, dem.shape[1], dem.shape[0], "Float32", geotransform=(100.0, 30.0, 0.0, 900.0, 0.0, -30.0))
    ds.GetRasterBand(1).WriteArray(dem)
    ds.GetRasterBand(1).SetNoDataValue(synth.NODATA)
    ds.FlushCache()
    allocs, pitched = [], dev.pitched

    def spy(rows, cols, dtype, device):  # sees every pitched buffer, the re-pitch copies of device.py's calls included
        allocs.append((rows, cols, dtype))
        return pitched(rows, cols, dtype, device)

    monkeypatch.setattr(dev, "pitched", spy)
    rep = stream_routing(src, str(tmp_path / "fdr_s.tif"), str(tmp_path / "fac_s.tif"), band_rows=band_rows)
    assert rep["rows"] == 333 and rep["bands"] == -(-333 // min(band_rows, 333)) and rep["wall_s"] > 0
    # the device DEM with its halo rows and the codes; no band of the stencil was copied to meet the TMA contract
    assert allocs == [(335, 257, torch.float32), (333, 257, torch.uint8)]
    whole = flow_routing_for_raster(dem, synth.NODATA)
    want_fdr = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1]
    want_fac = oracle.flow_accumulation(np.ascontiguousarray(want_fdr))
    for tag, want, plain, nd in (("fdr", want_fdr, whole[0], FLOW_DIRECTION_NODATA),
                                 ("fac", want_fac, whole[1], FLOW_ACCUMULATION_NODATA)):
        s_ds = open_raster(str(tmp_path / f"{tag}_s.tif"))
        got = s_ds.GetRasterBand(1).ReadAsArray()
        assert np.array_equal(got, want), tag
        assert np.array_equal(got, plain), tag
        assert s_ds.GetRasterBand(1).GetNoDataValue() == nd
        assert s_ds.GetGeoTransform() == (100.0, 30.0, 0.0, 900.0, 0.0, -30.0)


def test_streamed_direction_only_and_accumulation_only(tmp_path):
    from overflow_b200.streaming import stream_accumulation, stream_routing

    dem = synth.terraced(200, 130, seed=3)
    src = str(tmp_path / "dem.tif")
    ds = create_raster(src, dem.shape[1], dem.shape[0], "Float32")
    ds.GetRasterBand(1).WriteArray(dem)
    ds.GetRasterBand(1).SetNoDataValue(synth.NODATA)
    ds.FlushCache()
    fdr_path, fac_path, fac2_path = str(tmp_path / "fdr.tif"), str(tmp_path / "fac.tif"), str(tmp_path / "fac2.tif")
    stream_routing(src, fdr_path, None, band_rows=33)
    want_fdr = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1]
    assert np.array_equal(open_raster(fdr_path).GetRasterBand(1).ReadAsArray(), want_fdr)
    rep = stream_accumulation(fdr_path, fac_path, band_rows=40)
    want_fac = oracle.flow_accumulation(np.ascontiguousarray(want_fdr))
    assert np.array_equal(open_raster(fac_path).GetRasterBand(1).ReadAsArray(), want_fac)
    assert rep["h2d_bytes"] == dem.size and rep["d2h_bytes"] == dem.size * 8
    stream_routing(src, None, fac2_path, band_rows=64)
    assert np.array_equal(open_raster(fac2_path).GetRasterBand(1).ReadAsArray(), want_fac)


def test_streamed_driver_refuses_what_it_cannot_do(tmp_path):
    from overflow_b200.streaming import stream_routing

    src = str(tmp_path / "dem64.tif")
    ds = create_raster(src, 8, 8, "Float64")
    ds.GetRasterBand(1).WriteArray(np.zeros((8, 8)))
    ds.GetRasterBand(1).SetNoDataValue(-1)
    ds.FlushCache()
    with pytest.raises(TypeError):
        stream_routing(src, str(tmp_path / "o.tif"), None)
    with pytest.raises(ValueError):
        stream_routing(src, None, None)


def _write_raster(path, arr, dtype_name, nodata):
    ds = create_raster(path, arr.shape[1], arr.shape[0], dtype_name)
    ds.GetRasterBand(1).WriteArray(arr)
    ds.GetRasterBand(1).SetNoDataValue(nodata)
    ds.FlushCache()
    return path


def _pipeline_threads():
    return [t.name for t in threading.enumerate() if t.name.startswith("ofl-")]


@pytest.mark.parametrize("input_kind", ["dem", "codes"])
def test_streamed_write_failure_is_raised(tmp_path, monkeypatch, input_kind):
    """An output band whose second WriteArray fails (a full disk, say), with more bands than ring slots: the
    driver raises that error and leaves no pipeline thread behind, instead of waiting for a buffer forever."""
    from overflow_b200.streaming import stream_accumulation, stream_routing
    from overflow_b200.util import raster

    dem = synth.fractal(60, 50, beta=2.0, seed=4)
    fdr = np.ascontiguousarray(oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1])
    dem_path = _write_raster(str(tmp_path / "dem.tif"), dem, "Float32", synth.NODATA)
    fdr_path = _write_raster(str(tmp_path / "fdr.tif"), fdr, "Byte", FLOW_DIRECTION_NODATA)
    disk_full = OSError(28, "No space left on device")

    class Band:
        def __init__(self, band):
            self.band, self.writes = band, 0

        def __getattr__(self, name):
            return getattr(self.band, name)

        def WriteArray(self, *args, **kwargs):
            self.writes += 1
            if self.writes == 2:
                time.sleep(0.2)  # fails late: the driver is waiting for a free buffer by then
                raise disk_full
            return self.band.WriteArray(*args, **kwargs)

    class Dataset:
        def __init__(self, ds):
            self.ds = ds

        def __getattr__(self, name):
            return getattr(self.ds, name)

        def GetRasterBand(self, i):
            return Band(self.ds.GetRasterBand(i))

    create = raster.create_raster
    monkeypatch.setattr(raster, "create_raster", lambda *a, **k: Dataset(create(*a, **k)))
    outs = str(tmp_path / "fdr_s.tif"), str(tmp_path / "fac_s.tif")
    if input_kind == "dem":
        run = lambda: stream_routing(dem_path, *outs, band_rows=7, ring=2)  # noqa: E731
    else:
        run = lambda: stream_accumulation(fdr_path, outs[1], band_rows=7, ring=2)  # noqa: E731
    raised = []

    def call():
        try:
            run()
        except BaseException as e:  # noqa: BLE001 -- checked below
            raised.append(e)

    caller = threading.Thread(target=call, daemon=True)
    caller.start()
    caller.join(timeout=120)
    assert not caller.is_alive(), "the driver still waits 120 s after a failed write"
    assert raised == [disk_full]
    assert _pipeline_threads() == []


def test_streamed_accumulation_raises_on_a_cycle(tmp_path):
    from overflow_b200 import OverflowB200Error, _native
    from overflow_b200.streaming import stream_accumulation

    fdr = np.full((80, 80), 8, dtype=np.uint8)
    fdr[10, 10], fdr[10, 11] = 0, 4  # east and west: two cells pointing at each other
    src = _write_raster(str(tmp_path / "fdr.tif"), fdr, "Byte", FLOW_DIRECTION_NODATA)
    with pytest.raises(OverflowB200Error) as e:
        stream_accumulation(src, str(tmp_path / "fac.tif"), band_rows=16)
    assert e.value.status == _native.OFL_ERR_CYCLE
    assert _pipeline_threads() == []


def test_streamed_routing_frees_the_dem_before_the_accumulation(tmp_path):
    """The DEM (4 B/cell) is not held next to the codes, the counts and the accumulation workspace."""
    import torch

    from overflow_b200 import _native, device as dev
    from overflow_b200.streaming import stream_routing

    rows = cols = 2048
    dem = dev.synth_dem(rows, cols, seed=3, kind=0, holes_permille=5).cpu().numpy()
    src = _write_raster(str(tmp_path / "dem.tif"), dem, "Float32", -9999.0)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    stream_routing(src, str(tmp_path / "fdr.tif"), str(tmp_path / "fac.tif"))
    peak = torch.cuda.max_memory_allocated() - before
    cells = rows * cols
    accumulation = cells + cells * 8 + int(_native.lib().ofl_accumulation_workspace_bytes(rows, cols))
    dem_with_halo = (rows + 2) * cols * 4
    # held through the accumulation, the DEM made the peak accumulation + dem_with_halo
    assert peak < accumulation + dem_with_halo - 3 * cells, (peak, accumulation, dem_with_halo)


def test_flow_accumulation_cli_tiled(tmp_path):
    """--tile_size: the raster goes through the device in rectangular tiles (SURVEY 8f rank 3); same file."""
    dem = synth.punch_holes(synth.fractal(300, 260, beta=2.0, seed=25), frac=0.02, seed=26)
    fdr = np.ascontiguousarray(oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1])
    src, out = str(tmp_path / "fdr.tif"), str(tmp_path / "fac.tif")
    ds = create_raster(src, fdr.shape[1], fdr.shape[0], "Byte")
    ds.GetRasterBand(1).WriteArray(fdr)
    ds.GetRasterBand(1).SetNoDataValue(FLOW_DIRECTION_NODATA)
    ds.FlushCache()
    result = click.testing.CliRunner().invoke(
        flow_accumulation_cli, ["--input_file", src, "--output_file", out, "--tile_size", "128"])
    assert result.exit_code == 0, result.output
    band = open_raster(out).GetRasterBand(1)
    assert np.array_equal(band.ReadAsArray(), oracle.flow_accumulation(fdr))
    assert band.GetNoDataValue() == FLOW_ACCUMULATION_NODATA
