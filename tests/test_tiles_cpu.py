"""CPU tests of the rectangular-tile driver (overflow_b200/tiles.py, SURVEY 8f rank 3): the host-side consumer -- the
graph of all tiles' perimeter cells -- with a stand-in producer made of the CPU oracle.  The shipped producer is CUDA
only (tests/test_gpu_tiles.py)."""
import numpy as np
import pytest

import oracle
from oracle import synth
from overflow_b200 import tiles

DY = [0, -1, -1, -1, 0, 1, 1, 1]
DX = [1, 1, 0, -1, -1, -1, 0, 1]


class OracleTileEngine:
    """Same interface as tiles.CudaTileEngine: tile-local counts and perimeter links from the oracle's restatement of
    single_tile_flow_accumulation; inflow pushed down the paths cell by cell."""

    def accumulate(self, fdr, inflow=None, want_links=True):
        fdr = np.ascontiguousarray(fdr, dtype=np.uint8)
        h, w = fdr.shape
        fac, dense = oracle.single_tile_flow_accumulation(fdr)
        pr, pc = tiles.perimeter_cells(h, w)
        if inflow is not None:
            for k in np.nonzero(inflow)[0]:
                y, x, j = int(pr[k]), int(pc[k]), int(inflow[k])
                while True:
                    fac[y, x] += j
                    code = int(fdr[y, x])
                    if code >= 8:
                        break
                    ny, nx = y + DY[code], x + DX[code]
                    if not (0 <= ny < h and 0 <= nx < w) or fdr[ny, nx] == 9:
                        break
                    y, x = ny, nx
        return fac, (dense[pr, pc].copy() if want_links else None)


def codes_of(dem):
    return np.ascontiguousarray(oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1])


def dems():
    yield "fractal", synth.punch_holes(synth.fractal(150, 170, beta=2.5, seed=3), frac=0.03, seed=4)
    yield "terraced", synth.terraced(128, 96, seed=2)
    yield "tilted_se", synth.tilted_plane(96, 120)
    yield "tilted_nw", synth.tilted_plane(96, 120, a=-1.0, b=-0.5)
    yield "serpentine", oracle.synth_dem(97, 83, kind=3)
    yield "diagonal", (np.add.outer(np.arange(90), np.arange(110)) * -1.0).astype(np.float32)  # flows SE across tile corners


def test_perimeter_order_matches_the_reference_function():
    from overflow_b200.flow_accumulation import perimeter_indices

    for shape in [(1, 1), (1, 5), (5, 1), (2, 2), (3, 7), (7, 3), (64, 64)]:
        pr, pc = tiles.perimeter_cells(*shape)
        assert list(zip(pr.tolist(), pc.tolist())) == [tuple(x) for x in perimeter_indices(shape)]
        rank = tiles.perimeter_rank(pr, pc, *shape)
        for k in range(len(pr)):  # the rank of a cell is its first listing
            assert (pr[rank[k]], pc[rank[k]]) == (pr[k], pc[k]) and rank[k] <= k


@pytest.mark.parametrize("name,dem", list(dems()), ids=[n for n, _ in dems()])
@pytest.mark.parametrize("tile", [(64, 64), (50, 70), (33, 200), (200, 29), (1000, 1000), (1, 40), (17, 1)])
def test_tiled_accumulation_equals_whole_raster(name, dem, tile):
    fdr = codes_of(dem)
    want = oracle.flow_accumulation(fdr)
    rows, cols = fdr.shape
    if tile[0] * tile[1] < 200 and rows * cols > 12000:
        fdr, want = fdr[:40, :60].copy(), None  # thin tiles: keep the python stand-in quick
        want = oracle.flow_accumulation(fdr)
        rows, cols = fdr.shape
    got = np.full((rows, cols), -7, dtype=np.int64)

    def write_window(r0, c0, fac):
        got[r0 : r0 + fac.shape[0], c0 : c0 + fac.shape[1]] = fac

    n = tiles.flow_accumulation_tiled(lambda r0, r1, c0, c1: fdr[r0:r1, c0:c1], write_window, rows, cols, tile[0],
                                      tile[1], engine=OracleTileEngine())
    assert n == len(tiles.tile_grid(rows, cols, *tile))
    assert np.array_equal(got, want)


def test_cycle_across_tiles_is_reported():
    from overflow_b200 import _native

    fdr = np.full((4, 8), 8, dtype=np.uint8)
    fdr[1, 3], fdr[1, 4] = 0, 4  # (1,3) flows east into (1,4), which flows back west: a cycle across the tile boundary
    with pytest.raises(_native.OverflowB200Error) as ei:
        tiles.flow_accumulation_tiled(lambda r0, r1, c0, c1: fdr[r0:r1, c0:c1], lambda *a: None, 4, 8, 4, 4,
                                      engine=OracleTileEngine())
    assert ei.value.status == _native.OFL_ERR_CYCLE


def test_code_outside_0_255_is_refused():
    fdr = np.full((4, 8), 8, dtype=np.int64)
    fdr[2, 5] = 265  # would wrap to 9 (NODATA) as uint8
    with pytest.raises(ValueError, match="0..255"):
        tiles.flow_accumulation_tiled(lambda r0, r1, c0, c1: fdr[r0:r1, c0:c1], lambda *a: None, 4, 8, 4, 4,
                                      engine=OracleTileEngine())


def test_tiled_file_driver(tmp_path):
    from overflow_b200.util.raster import create_raster, open_raster

    fdr = codes_of(synth.punch_holes(synth.fractal(130, 90, beta=2.0, seed=8), frac=0.02, seed=9))
    src = str(tmp_path / "fdr.tif")
    ds = create_raster(src, 90, 130, "Byte")
    ds.GetRasterBand(1).WriteArray(fdr)
    ds.GetRasterBand(1).SetNoDataValue(9)
    ds.FlushCache()
    out = str(tmp_path / "fac.tif")
    assert tiles.flow_accumulation_file_tiled(src, out, 48, 40, engine=OracleTileEngine()) == 9
    band = open_raster(out).GetRasterBand(1)
    assert np.array_equal(band.ReadAsArray(), oracle.flow_accumulation(fdr)) and band.GetNoDataValue() == -9999
