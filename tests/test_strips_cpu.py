"""CPU tests of the row-strip host logic: partitioning, loop-back exchange and a world_size-2 gloo run.

The compute engine here is tests/strip_numpy_engine.py (oracle-based stand-in); the shipped engine is
CUDA only.  What is under test is overflow_b200.strips: halo exchange, all-gather, phase ordering."""
import os
import socket

import numpy as np
import pytest
import torch

import oracle
from oracle import synth
from overflow_b200 import strips
from strip_numpy_engine import NumpyStripEngine


def test_partition_rows():
    assert strips.partition_rows(65536, 8) == [(i * 8192, (i + 1) * 8192) for i in range(8)]
    p = strips.partition_rows(1000, 3)
    assert p[0][0] == 0 and p[-1][1] == 1000
    assert all(a % 64 == 0 for a, _ in p) and all(p[i][1] == p[i + 1][0] for i in range(2))
    assert strips.partition_rows(321, 4) == [(0, 128), (128, 192), (192, 256), (256, 321)]
    with pytest.raises(ValueError):
        strips.partition_rows(200, 4)


def whole_raster_oracle(dem):
    fdr = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1].copy()
    return fdr, oracle.flow_accumulation(fdr)


def make_dems():
    yield "fractal", synth.punch_holes(synth.fractal(200, 90, beta=2.5, seed=3), frac=0.02, seed=4)
    yield "tilted_south", synth.tilted_plane(192, 40)
    yield "tilted_north", synth.tilted_plane(192, 40, a=-1.0, b=0.5)
    yield "serpentine", synth.serpentine(193, 31)


@pytest.mark.parametrize("name,dem", list(make_dems()), ids=[n for n, _ in make_dems()])
@pytest.mark.parametrize("world", [1, 2, 3])
def test_in_process_strips_match_whole_raster(name, dem, world):
    rows, cols = dem.shape
    pipes = [strips.StripPipeline(rows, cols, r, world, nodata=synth.NODATA, engine=NumpyStripEngine())
             for r in range(world)]
    for p in pipes:
        p.load_dem(dem[p.r0 : p.r1])
    strips.step_in_process(pipes)
    want_fdr, want_fac = whole_raster_oracle(dem)
    got_fdr = np.concatenate([p.fdr.numpy() for p in pipes])
    got_fac = np.concatenate([p.fac.numpy() for p in pipes])
    assert np.array_equal(got_fdr, want_fdr)
    assert np.array_equal(got_fac, want_fac)
    # the recurrence check across strip boundaries: clean on the result, and it sees a wrong boundary count
    assert strips.check_in_process(pipes) == 0
    if world > 1:
        pipes[1].fac[0, cols // 2] += 1
        assert strips.check_in_process(pipes) >= 1


def test_record_layout_matches_library():
    from overflow_b200 import _native, build

    build.build()
    for cols in (1, 7, 64, 1000, 65536):
        assert strips.record_bytes(cols) == _native.lib().ofl_strip_record_bytes(cols)
    rec = torch.zeros((3, strips.record_bytes(10)), dtype=torch.uint8)
    floc, slink, bcode = strips.record_views(rec, 10)
    assert floc.shape == slink.shape == bcode.shape == (3, 2, 10)
    floc[1, 1, 9] = -5
    slink[2, 0, 0] = 77
    bcode[0, 1, 3] = 9
    one = strips.record_views(rec[1], 10)[0]
    assert one.shape == (2, 10) and int(one[1, 9]) == -5
    assert int(rec[2, 160:164].view(torch.int32)[0]) == 77 and int(rec[0, 240 + 13]) == 9


def _gloo_worker(rank, world, port, dem, out_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rows, cols = dem.shape
        p = strips.StripPipeline(rows, cols, rank, world, nodata=synth.NODATA, engine=NumpyStripEngine())
        p.load_dem(dem[p.r0 : p.r1])
        p.step()
        bad = torch.tensor([p.check()])
        dist.all_reduce(bad)
        assert int(bad.item()) == 0
        np.save(os.path.join(out_dir, f"fdr{rank}.npy"), p.fdr.numpy())
        np.save(os.path.join(out_dir, f"fac{rank}.npy"), p.fac.numpy())
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_gloo_world_size_2(tmp_path):
    import torch.multiprocessing as mp

    dem = synth.punch_holes(synth.fractal(160, 70, beta=3.0, seed=8), frac=0.02, seed=9)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_gloo_worker, args=(2, port, dem, str(tmp_path)), nprocs=2, join=True)
    want_fdr, want_fac = whole_raster_oracle(dem)
    got_fdr = np.concatenate([np.load(tmp_path / f"fdr{r}.npy") for r in range(2)])
    got_fac = np.concatenate([np.load(tmp_path / f"fac{r}.npy") for r in range(2)])
    assert np.array_equal(got_fdr, want_fdr)
    assert np.array_equal(got_fac, want_fac)


# ---- out of core: the same strip structure through one engine, strip by strip (SURVEY 8f rank 3)
def test_strip_bounds():
    assert strips.strip_bounds(200, 64) == [(0, 64), (64, 128), (128, 200)]  # 8 leftover rows join the last strip
    assert strips.strip_bounds(256, 64) == [(0, 64), (64, 128), (128, 192), (192, 256)]
    assert strips.strip_bounds(40, 64) == [(0, 40)]
    assert strips.strip_bounds(128, 128) == [(0, 128)]
    with pytest.raises(ValueError):
        strips.strip_bounds(200, 100)


@pytest.mark.parametrize("name,dem", list(make_dems()), ids=[n for n, _ in make_dems()])
@pytest.mark.parametrize("strip_rows", [64, 128])
def test_out_of_core_matches_whole_raster(name, dem, strip_rows):
    want_fdr, want_fac = whole_raster_oracle(dem)
    rows, cols = want_fdr.shape
    got = np.full((rows, cols), -7, dtype=np.int64)
    reads = []

    def read_rows(r0, r1):
        reads.append((r0, r1))
        return want_fdr[r0:r1]

    def write_rows(r0, fac):
        got[r0 : r0 + len(fac)] = fac

    n = strips.flow_accumulation_out_of_core(read_rows, write_rows, rows, cols, strip_rows, engine=NumpyStripEngine())
    assert n == len(strips.strip_bounds(rows, strip_rows)) and len(reads) == 2 * n  # every strip is read twice
    assert np.array_equal(got, want_fac)


def test_out_of_core_refuses_a_code_outside_0_255():
    fdr = np.full((130, 20), 8, dtype=np.int64)
    fdr[100, 7] = 265  # would wrap to 9 (NODATA) as uint8
    with pytest.raises(ValueError, match="0..255"):
        strips.flow_accumulation_out_of_core(lambda r0, r1: fdr[r0:r1], lambda r0, fac: None, 130, 20, 64,
                                             engine=NumpyStripEngine())


def test_out_of_core_file_driver(tmp_path):
    from overflow_b200.util.raster import create_raster, open_raster

    dem = synth.punch_holes(synth.fractal(150, 70, beta=2.5, seed=8), frac=0.02, seed=9)
    want_fdr, want_fac = whole_raster_oracle(dem)
    src = str(tmp_path / "fdr.tif")
    ds = create_raster(src, 70, 150, "Byte")
    ds.GetRasterBand(1).WriteArray(want_fdr)
    ds.GetRasterBand(1).SetNoDataValue(9)
    ds.FlushCache()
    out = str(tmp_path / "fac.tif")
    assert strips.flow_accumulation_file_out_of_core(src, out, 64, engine=NumpyStripEngine()) == 2  # 64 + 86 rows
    band = open_raster(out).GetRasterBand(1)
    assert np.array_equal(band.ReadAsArray(), want_fac) and band.GetNoDataValue() == -9999
