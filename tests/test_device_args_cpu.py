"""CPU tests of the argument checks every overflow_b200.device call runs before its tensors reach the C ABI: dtype,
shape, device, column stride, row pitch and workspace size.  The checks come before the library is initialised, so
they run on CPU tensors; a CPU tensor that passes them is refused as not being on a CUDA device."""
import pytest
import torch

from overflow_b200 import device as dev

CPU = torch.device("cpu")


@pytest.mark.parametrize("t,message", [
    (torch.zeros((4, 8), dtype=torch.float64), "float32"),
    (torch.zeros((32,), dtype=torch.float32), "2-D"),
    (torch.zeros((2, 4, 8), dtype=torch.float32), "2-D"),
    (torch.zeros((4, 16), dtype=torch.float32)[:, ::2], "unit column stride"),
    (torch.zeros((8, 4), dtype=torch.float32).t(), "unit column stride"),
], ids=["dtype", "1-D", "3-D", "strided", "transposed"])
def test_input_refuses_what_the_library_would_misread(t, message):
    with pytest.raises(ValueError, match=message):
        dev._input("dem", t, torch.float32, repitch=True)


@pytest.mark.parametrize("t", [
    torch.zeros((4, 8), dtype=torch.uint8),
    torch.zeros((3, 4), dtype=torch.uint8).t()[:, :1],  # one column: its column stride addresses nothing
], ids=["dense", "one-column"])
def test_input_that_passes_the_checks_still_needs_a_cuda_tensor(t):
    with pytest.raises(ValueError, match="CUDA tensor"):
        dev._input("fdr", t, torch.uint8)


def _bad_outputs():
    yield "dtype", torch.zeros((4, 8), dtype=torch.int32), {}, "int64 tensor of shape"
    yield "shape", torch.zeros((4, 7), dtype=torch.int64), {}, "shape"
    yield "1-D", torch.zeros((32,), dtype=torch.int64), {}, "shape"
    yield "not a tensor", [[0] * 8] * 4, {}, "shape"
    yield "device", torch.zeros((4, 8), dtype=torch.int64, device="meta"), {}, "must live on cpu"
    yield "stride", torch.zeros((4, 16), dtype=torch.int64)[:, ::2], {}, "unit column stride"
    yield "pitch below width", torch.zeros(64, dtype=torch.int64).as_strided((4, 8), (4, 1)), {}, "row pitch 4"
    yield "pitch multiple", torch.zeros((4, 10), dtype=torch.int64)[:, :8], {"align": 4}, "multiple of 4"
    yield "dense", torch.zeros((4, 16), dtype=torch.int64)[:, :8], {"dense": True}, "equal to 8"


@pytest.mark.parametrize("name,t,kw,message", list(_bad_outputs()), ids=[c[0] for c in _bad_outputs()])
def test_output_refuses_what_the_library_would_misread(name, t, kw, message):
    with pytest.raises(ValueError, match=message):
        dev._output("out", t, torch.int64, (4, 8), CPU, **kw)
    with pytest.raises(ValueError, match=message):
        dev._check_raster("fac", t, torch.int64, (4, 8), CPU, **kw)


def test_output_accepts_pitched_and_degenerate_layouts():
    padded = torch.zeros((4, 12), dtype=torch.uint8)[:, :8]
    assert dev._output("out", padded, torch.uint8, (4, 8), CPU, 4) is padded
    one_row = torch.zeros(64, dtype=torch.int64).as_strided((1, 8), (3, 1))  # one row: its pitch addresses nothing
    assert dev._output("out", one_row, torch.int64, (1, 8), CPU, 16, dense=True) is one_row
    one_col = torch.zeros((3, 4), dtype=torch.int64).t()[:, :1]
    assert dev._check_raster("labels", one_col, torch.int64, (4, 1), CPU) is one_col
    dense = torch.zeros((4, 8), dtype=torch.int32)
    assert dev._output("flat_mask", dense, torch.int32, (4, 8), CPU, dense=True) is dense


@pytest.mark.parametrize("dtype,pitch", [(torch.uint8, 32), (torch.float32, 20), (torch.int64, 17), (torch.int8, 17)])
def test_new_outputs_get_the_library_pitch(dtype, pitch):
    """Codes get 16-byte row pitches and DEMs 4-cell ones, as TMA reads them; other rasters are dense."""
    t = dev._output("out", None, dtype, (3, 17), CPU)
    assert t.dtype == dtype and tuple(t.shape) == (3, 17) and t.stride() == (pitch, 1)
    assert dev.pitched(3, 17, dtype, CPU).stride() == (pitch, 1)


@pytest.fixture(scope="module")
def library():
    from overflow_b200 import _native, build

    build.build()
    return _native.lib()


@pytest.mark.parametrize("kind,query", [("accumulation", "ofl_accumulation_workspace_bytes"),
                                        ("basins", "ofl_basins_workspace_bytes"),
                                        ("flats", "ofl_flats_workspace_bytes"),
                                        ("pits", "ofl_pits_workspace_bytes"),
                                        ("strip", "ofl_strip_workspace_bytes"),
                                        ("strip_boundary", "ofl_strip_boundary_workspace_bytes")])
def test_workspace_is_sized_by_the_library_and_checked(library, kind, query):
    rows, cols = 4, 300
    need = int(getattr(library, query)(rows, cols))
    assert need > 0
    ws = dev._workspace(kind, rows, cols, CPU)
    assert ws.dtype == torch.uint8 and tuple(ws.shape) == (need,)
    assert dev._workspace(kind, rows, cols, CPU, ws) is ws
    for bad, message in ((torch.zeros(need - 1, dtype=torch.uint8), f"holds {need - 1} bytes, {need} needed"),
                         (torch.zeros(need, dtype=torch.int8), "1-D uint8"),
                         (torch.zeros((1, need), dtype=torch.uint8), "1-D uint8"),
                         (torch.zeros(2 * need, dtype=torch.uint8)[::2], "contiguous"),
                         (torch.zeros(need, dtype=torch.uint8, device="meta"), "must live on cpu")):
        with pytest.raises(ValueError, match=message):
            dev._workspace(kind, rows, cols, CPU, bad)


def test_calls_refuse_cpu_tensors_before_the_library():
    """A CPU tensor never reaches the library, the strip calls included."""
    dem, fdr, fac = torch.zeros((6, 8)), torch.zeros((6, 8), dtype=torch.uint8), torch.zeros((4, 8), dtype=torch.int64)
    calls = [
        lambda: dev.flow_direction(dem, -9999.0),
        lambda: dev.flow_routing(dem, -9999.0),
        lambda: dev.flow_accumulation(fdr),
        lambda: dev.check_accumulation(fdr, fac),
        lambda: dev.label_basins(fdr),
        lambda: dev.resolve_flats(dem, fdr),
        lambda: dev.breach_single_cell_pits(dem, -9999.0),
        lambda: dev.synth_dem(6, 8, out=dem),
        lambda: dev.strip_accum_local(fdr, True, False, fac, None, None),
        lambda: dev.strip_check_accumulation(fdr, fac, None, None),
    ]
    for call in calls:
        with pytest.raises(ValueError, match="CUDA tensor"):
            call()
