"""GPU: host-memory calls stage their rasters through library-owned device buffers.  A call returns only once every
copy it started has finished, whether it succeeds or fails, and a failed call leaves nothing in the staging buffers
that changes the result of the next call."""
import numpy as np
import pytest

import oracle
from oracle import synth
from overflow_b200 import OverflowB200Error, _native, tiles
from overflow_b200.flow_accumulation import flow_accumulation_for_raster, single_tile_flow_accumulation
from test_tiles_cpu import OracleTileEngine

pytestmark = pytest.mark.gpu

OFL_ERR_WORKSPACE = -6


def test_failed_call_returns_with_no_copy_in_flight():
    """A caller workspace one byte too small is refused before the 64 MB upload of the pinned codes is queued, so
    nothing the call started is in flight when it returns and the caller may free or reuse its buffers at once."""
    import torch

    rows = cols = 8192
    _native.init(torch.cuda.current_device())
    lib = _native.lib()
    codes = torch.full((rows, cols), 8, dtype=torch.uint8).pin_memory()
    fac = np.empty((rows, cols), dtype=np.int64)
    need = int(lib.ofl_accumulation_workspace_bytes(rows, cols))
    work = torch.empty(need - 1, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    rc = lib.ofl_flow_accumulation_u8(codes.data_ptr(), rows, cols, cols, fac.ctypes.data, cols, None, work.data_ptr(),
                                      need - 1, _native.OFL_MEM_HOST, stream.cuda_stream)
    idle = stream.query()
    assert rc == OFL_ERR_WORKSPACE
    assert idle


def test_call_failing_after_its_upload_returns_with_no_copy_in_flight():
    """A cyclic raster fails only once the 64 MB of pinned codes are on the device and the accumulation has run; the
    call still waits for everything it started before it returns."""
    import torch

    rows = cols = 8192
    _native.init(torch.cuda.current_device())
    lib = _native.lib()
    codes = torch.full((rows, cols), 8, dtype=torch.uint8).pin_memory()
    codes[rows // 2, cols // 2], codes[rows // 2, cols // 2 + 1] = 0, 4  # two cells pointing at each other
    fac = torch.empty((rows, cols), dtype=torch.int64).pin_memory()
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    rc = lib.ofl_flow_accumulation_u8(codes.data_ptr(), rows, cols, cols, fac.data_ptr(), cols, None, None, 0,
                                      _native.OFL_MEM_HOST, stream.cuda_stream)
    idle = stream.query()
    assert rc == _native.OFL_ERR_CYCLE
    assert idle


ROUTES = ["flow_accumulation_for_raster", "single_tile_flow_accumulation", "tile_engine_with_inflow"]


def route(name, fdr):
    """(run, want) of one host accumulation route; the tile engine gets inflow on every first-listed perimeter cell
    that is not NODATA."""
    if name == "flow_accumulation_for_raster":
        return (lambda f: flow_accumulation_for_raster(f, with_links=True),
                lambda f: (oracle.flow_accumulation(f), oracle.links_perimeter(f)[1]))
    if name == "single_tile_flow_accumulation":
        return single_tile_flow_accumulation, oracle.single_tile_flow_accumulation
    h, w = fdr.shape
    pr, pc = tiles.perimeter_cells(h, w)
    inflow = np.random.default_rng(7).integers(1, 1000, len(pr), dtype=np.int64)
    inflow[(tiles.perimeter_rank(pr, pc, h, w) != np.arange(len(pr))) | (fdr[pr, pc] == 9)] = 0
    return (lambda f: tiles.CudaTileEngine().accumulate(f, inflow, True),
            lambda f: OracleTileEngine().accumulate(f, inflow, True))


@pytest.mark.parametrize("name", ROUTES)
def test_cycle_then_valid_raster_through_the_same_route(name):
    dem = synth.punch_holes(synth.fractal(300, 333, beta=2.5, seed=12), frac=0.02, seed=13)
    fdr = np.ascontiguousarray(oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1])
    cyclic = fdr.copy()
    cyclic[150, 166], cyclic[150, 167] = 0, 4  # two cells pointing at each other
    run, want = route(name, fdr)
    with pytest.raises(OverflowB200Error) as e:
        run(cyclic)
    assert e.value.status == _native.OFL_ERR_CYCLE
    # same shape: the valid raster reuses the staging buffers the failed call left behind
    for got, expected in zip(run(fdr), want(fdr)):
        assert np.array_equal(got, expected)
