"""Device-resident entry points: torch CUDA tensors in, torch CUDA tensors out.

PyTorch is only the owner of device memory and streams here; every kernel is in
liboverflow_b200.  Calls are enqueued on torch's current stream.

Every library call on torch tensors is made from this module, so it alone knows how a tensor meets the C ABI: the
argument order, unit column stride, and the 16-byte base and row pitch the TMA tensor maps want (16 codes, 4 DEM cells).
"""
import ctypes

import torch

from . import _native


def _stream(t):
    """torch's current stream on the tensor's device (not on whatever device happens to be current)."""
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _init_for(t: torch.Tensor):
    if not t.is_cuda:
        raise ValueError("expected a CUDA tensor (there is no CPU fallback)")
    _native.init(t.device.index if t.device.index is not None else torch.cuda.current_device())


# Codes and DEMs get 16-byte row pitches: the stencil and the accumulation read them through TMA tensor maps, which a
# dense tensor of odd width does not satisfy.  Other rasters are dense.
_PITCH = {torch.uint8: 16, torch.float32: 4}


def pitched(rows, cols, dtype, device):
    """rows x cols view of a new buffer with the row pitch the library wants for `dtype`."""
    align = _PITCH.get(dtype, 1)
    return torch.empty((rows, (cols + align - 1) // align * align), dtype=dtype, device=device)[:, :cols]


def _input(name, t, dtype, repitch=False):
    """`t`, a raster the call reads, checked, with the library initialised on its device.  With `repitch`, a raster
    whose row pitch or base address does not meet the TMA contract comes back as a pitched copy.  A one-column
    raster may have any column stride: it never addresses memory."""
    if t.dtype != dtype or t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise ValueError(f"{name} must be a 2-D {dtype} tensor with unit column stride")
    _init_for(t)
    if repitch and t.numel() and (t.stride(0) % _PITCH[dtype] or t.data_ptr() % 16):
        t = pitched(t.shape[0], t.shape[1], dtype, t.device).copy_(t)
    return t


def _check_raster(name, t, dtype, shape, device, align=1, dense=False):
    """Raw pointers of `t` go straight into the C ABI: refuse anything it would mis-read.  The row pitch must be a
    multiple of `align` elements, or with `dense` equal to the width (calls that take packed rows)."""
    if not isinstance(t, torch.Tensor) or t.dtype != dtype or t.dim() != 2 or tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} must be a {dtype} tensor of shape {tuple(shape)}")
    if t.device != device:
        raise ValueError(f"{name} must live on {device}, not {t.device}")
    if t.shape[1] > 1 and t.stride(1) != 1:
        raise ValueError(f"{name} must have unit column stride")
    pitch, width = t.stride(0), t.shape[1]
    if t.shape[0] > 1 and (pitch < width or pitch % align or (dense and pitch != width)):
        want = f"equal to {width}" if dense else f">= {width} and a multiple of {align}"
        raise ValueError(f"{name}: row pitch {pitch} must be {want}")
    return t


def _output(name, t, dtype, shape, device, align=1, dense=False):
    """The caller's raster `t` for the call to write, checked as _check_raster does; or, when it is None, a new one."""
    if t is None:
        return pitched(*shape, dtype, device)
    return _check_raster(name, t, dtype, shape, device, align, dense)


def _workspace(kind, rows, cols, device, t=None):
    """The caller's workspace `t` for a rows x cols `kind` call, checked to hold ofl_<kind>_workspace_bytes(rows, cols)
    bytes; or, when it is None, a new one of that size."""
    need = int(getattr(_native.lib(), f"ofl_{kind}_workspace_bytes")(rows, cols))
    if t is None:
        return torch.empty((need,), dtype=torch.uint8, device=device)
    if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or t.dim() != 1 or not t.is_contiguous():
        raise ValueError("workspace must be a contiguous 1-D uint8 tensor")
    if t.device != device:
        raise ValueError(f"workspace must live on {device}, not {t.device}")
    if t.numel() < need:
        raise ValueError(f"workspace holds {t.numel()} bytes, {need} needed")
    return t


def synth_dem(rows, cols, *, row0=0, total_rows=None, seed=0, kind=0, relief=1000.0, holes_permille=0,
              nodata=-9999.0, device="cuda", out=None):
    """Seeded synthetic float32 DEM generated on the device (kind 0 fractal, 1 terraces, 2 tilted plane,
    3 walled serpentine: one channel of about rows * cols / 2 cells running east-west; 4 the same running north-south).

    Rows row0..row0+rows-1 of a raster with `total_rows` rows; rows outside [0,total_rows) are nodata
    (that is what a strip's halo row is at the raster top / bottom).  `out`: write into this tensor.
    """
    total_rows = rows if total_rows is None else total_rows
    dem = _output("out", out, torch.float32, (rows, cols), out.device if out is not None else device)
    _init_for(dem)
    _native.check(
        _native.lib().ofl_synth_dem_f32(
            dem.data_ptr(), rows, cols, dem.stride(0), row0, total_rows, seed, kind, relief, holes_permille, nodata,
            _stream(dem),
        )
    )
    return dem


def flow_direction(dem: torch.Tensor, nodata_value: float, *, mode="raster", out=None) -> torch.Tensor:
    """uint8 D8 codes of a float32 CUDA raster.

    mode "raster": whole raster, out-of-raster neighbours are nodata.
    mode "tile":   flow_direction_for_tile semantics (dem carries its ring; ring of the result is 9).
    mode "strip":  dem has 2 more rows than the result: halo rows above and below.
    """
    dem = _input("dem", dem, torch.float32, repitch=True)
    m = {"tile": _native.OFL_DIR_MODE_TILE, "raster": _native.OFL_DIR_MODE_RASTER, "strip": _native.OFL_DIR_MODE_STRIP}[mode]
    rows, cols = dem.shape
    if m == _native.OFL_DIR_MODE_STRIP:
        rows -= 2
    out = _output("out", out, torch.uint8, (rows, cols), dem.device, 4)
    _native.check(
        _native.lib().ofl_flow_direction_f32(
            dem.data_ptr(), rows, cols, dem.stride(0), float(nodata_value), out.data_ptr(), out.stride(0), m,
            _native.OFL_MEM_DEVICE, _stream(dem),
        )
    )
    return out


def accumulation_workspace(rows, cols, device="cuda") -> torch.Tensor:
    return _workspace("accumulation", rows, cols, device)


def flow_accumulation(fdr: torch.Tensor, *, out=None, workspace=None, with_links=False):
    """int64 upstream-cell counts of a uint8 CUDA flow-direction raster.

    Returns fac, or (fac, perim_links[n,2]) in perimeter_indices order when with_links.
    Synchronises the stream (the perimeter-graph solve reports convergence to the host).
    """
    fdr = _input("fdr", fdr, torch.uint8, repitch=True)
    rows, cols = fdr.shape
    out = _output("out", out, torch.int64, (rows, cols), fdr.device)
    workspace = _workspace("accumulation", rows, cols, fdr.device, workspace)
    links = None
    if with_links:
        n = int(_native.lib().ofl_perimeter_count(rows, cols))
        links = torch.empty((n, 2), dtype=torch.int64, device=fdr.device)
    _native.check(
        _native.lib().ofl_flow_accumulation_u8(
            fdr.data_ptr(), rows, cols, fdr.stride(0), out.data_ptr(), out.stride(0),
            links.data_ptr() if with_links else None, workspace.data_ptr(), workspace.numel(),
            _native.OFL_MEM_DEVICE, _stream(fdr),
        )
    )
    return (out, links) if with_links else out


def flow_routing(dem: torch.Tensor, nodata_value: float, *, out_fdr=None, out_fac=None, resolve_flats=False):
    """(fdr uint8, fac int64) of a float32 CUDA DEM in one library call (ofl_flow_routing_f32): the
    accumulation workspace is library-owned and cleared next to the stencil.  Synchronises the stream.

    resolve_flats=True runs the three steps as the reference orders them -- flow direction, flat resolution
    (fix_flats.py), accumulation -- with the codes resident on the device throughout.  The DEM must be free of
    pits then (the reference breaches them first): its d8_masked_flow_dirs points a pit at a neighbour, which can
    close a cycle, and a cyclic raster makes the accumulation raise OFL_ERR_CYCLE."""
    if resolve_flats:
        _input("dem", dem, torch.float32)
        if not dem.is_contiguous():
            raise ValueError("resolve_flats needs a contiguous DEM")
        if dem.shape[1] % 16:
            raise ValueError("resolve_flats needs a column count that is a multiple of 16 (dense codes, TMA pitch)")
        fdr = flow_direction(dem, nodata_value, out=out_fdr)
        fix_flats(dem, fdr)
        return fdr, flow_accumulation(fdr, out=out_fac)
    dem = _input("dem", dem, torch.float32, repitch=True)
    rows, cols = dem.shape
    out_fdr = _output("out_fdr", out_fdr, torch.uint8, (rows, cols), dem.device, 16)
    out_fac = _output("out_fac", out_fac, torch.int64, (rows, cols), dem.device)
    _native.check(
        _native.lib().ofl_flow_routing_f32(
            dem.data_ptr(), rows, cols, dem.stride(0), float(nodata_value), out_fdr.data_ptr(), out_fdr.stride(0),
            out_fac.data_ptr(), out_fac.stride(0), None, _native.OFL_MEM_DEVICE, _stream(dem),
        )
    )
    return out_fdr, out_fac


def check_accumulation(fdr: torch.Tensor, fac: torch.Tensor) -> int:
    """Number of cells violating the accumulation recurrence (0 proves fac exact on an acyclic raster)."""
    fdr = _input("fdr", fdr, torch.uint8)
    rows, cols = fdr.shape
    _check_raster("fac", fac, torch.int64, (rows, cols), fdr.device)
    n_bad = ctypes.c_int64(0)
    _native.check(
        _native.lib().ofl_check_accumulation_u8(
            fdr.data_ptr(), rows, cols, fdr.stride(0), fac.data_ptr(), fac.stride(0), ctypes.byref(n_bad),
            _native.OFL_MEM_DEVICE, _stream(fdr),
        )
    )
    return int(n_bad.value)


def basins_workspace(rows, cols, device="cuda") -> torch.Tensor:
    return _workspace("basins", rows, cols, device)


def _pour_indices(pour_points, fdr):
    """Row-major int64 cell indices on fdr's device of an (k, 2) array or tensor of (row, col); None when there are
    no pour points.  A point outside the raster raises ValueError (for a tensor this reads one flag back)."""
    if pour_points is None:
        return None
    rows, cols = fdr.shape
    if isinstance(pour_points, torch.Tensor):
        pp = pour_points.reshape(0, 2) if pour_points.numel() == 0 else pour_points
        if pp.dim() != 2 or pp.shape[1] != 2 or pp.dtype.is_floating_point or pp.dtype.is_complex or pp.dtype == torch.bool:
            raise ValueError("pour points must be an integer (k, 2) tensor of (row, col)")
        pp = pp.to(device=fdr.device, dtype=torch.int64)
        if bool(((pp[:, 0] < 0) | (pp[:, 0] >= rows) | (pp[:, 1] < 0) | (pp[:, 1] >= cols)).any()):
            raise ValueError(f"pour point outside the {rows} x {cols} raster")
        idx = (pp[:, 0] * cols + pp[:, 1]).contiguous()
    else:
        from .basins import pour_point_indices

        idx = torch.from_numpy(pour_point_indices(pour_points, (rows, cols))).to(fdr.device)
    return idx if idx.numel() else None


def label_basins(fdr: torch.Tensor, *, pour_points=None, out=None, workspace=None) -> torch.Tensor:
    """int64 basin labels of a uint8 CUDA flow-direction raster (overflow_b200.basins has the rules): the label of
    the outlet, or with pour points ((k, 2) of (row, col)) of the first pour point, that each cell's path reaches.
    Synchronises the stream (the call reports cycles and pour points outside the raster)."""
    fdr = _input("fdr", fdr, torch.uint8, repitch=True)
    rows, cols = fdr.shape
    idx = _pour_indices(pour_points, fdr)
    out = _output("out", out, torch.int64, (rows, cols), fdr.device)
    workspace = _workspace("basins", rows, cols, fdr.device, workspace)
    _native.check(
        _native.lib().ofl_label_basins_u8(
            fdr.data_ptr(), rows, cols, fdr.stride(0), idx.data_ptr() if idx is not None else None,
            0 if idx is None else idx.numel(), out.data_ptr(), out.stride(0), workspace.data_ptr(), workspace.numel(),
            _native.OFL_MEM_DEVICE, _stream(fdr),
        )
    )
    return out


def check_basins(fdr: torch.Tensor, labels: torch.Tensor, pour_points=None) -> int:
    """Number of cells breaking the basin labelling rule (0 proves the labels exact on an acyclic raster)."""
    fdr = _input("fdr", fdr, torch.uint8)
    rows, cols = fdr.shape
    _check_raster("labels", labels, torch.int64, (rows, cols), fdr.device)
    idx = _pour_indices(pour_points, fdr)
    n_bad = ctypes.c_int64(0)
    _native.check(
        _native.lib().ofl_check_basins_u8(
            fdr.data_ptr(), rows, cols, fdr.stride(0), idx.data_ptr() if idx is not None else None,
            0 if idx is None else idx.numel(), labels.data_ptr(), labels.stride(0), ctypes.byref(n_bad),
            _native.OFL_MEM_DEVICE, _stream(fdr),
        )
    )
    return int(n_bad.value)


def flats_workspace(rows, cols, device="cuda") -> torch.Tensor:
    return _workspace("flats", rows, cols, device)


def _flats_call(fix, dem, fdr, flat_mask, labels, workspace):
    """ofl_fix_flats_f32 when `fix`, else ofl_resolve_flats_f32: (flat_mask, labels, info).  Both take packed rows:
    every raster is dense."""
    _input("dem", dem, torch.float32)
    rows, cols = dem.shape
    _check_raster("dem", dem, torch.float32, (rows, cols), dem.device, dense=True)
    _check_raster("fdr", fdr, torch.uint8, (rows, cols), dem.device, dense=True)
    flat_mask = _output("flat_mask", flat_mask, torch.int32, (rows, cols), dem.device, dense=True)
    labels = _output("labels", labels, torch.int32, (rows, cols), dem.device, dense=True)
    workspace = _workspace("flats", rows, cols, dem.device, workspace)
    info = (ctypes.c_int64 * 5)()
    fn = _native.lib().ofl_fix_flats_f32 if fix else _native.lib().ofl_resolve_flats_f32
    _native.check(
        fn(dem.data_ptr(), fdr.data_ptr(), rows, cols, flat_mask.data_ptr(), labels.data_ptr(), info,
           workspace.data_ptr(), workspace.numel(), _native.OFL_MEM_DEVICE, _stream(dem))
    )
    return flat_mask, labels, [int(v) for v in info]


def resolve_flats(dem: torch.Tensor, fdr: torch.Tensor, *, workspace=None):
    """(flat_mask int32, labels int32, info) of a float32 CUDA DEM and its uint8 codes (ofl_resolve_flats_f32).
    info = [low edges, high edges, labels, away levels, towards levels].  Synchronises the stream."""
    return _flats_call(False, dem, fdr, None, None, workspace)


def fix_flats(dem: torch.Tensor, fdr: torch.Tensor, *, workspace=None, flat_mask=None, labels=None):
    """Rewrite the code-8 cells of `fdr` in place (resolve_flats + d8_masked_flow_dirs, ofl_fix_flats_f32).
    Returns (fdr, info).  Synchronises the stream."""
    return fdr, _flats_call(True, dem, fdr, flat_mask, labels, workspace)[2]


def breach_single_cell_pits(chunk: torch.Tensor, nodata_value: float, *, unsolved=None, workspace=None):
    """Breach the single-cell pits of a float32 CUDA chunk in place (ofl_breach_single_cell_pits_f32).
    Returns (unsolved int8 tensor, [pits found, pits left unsolved, rounds]).  Synchronises the stream."""
    chunk = _input("chunk", chunk, torch.float32)
    rows, cols = chunk.shape
    unsolved = _output("unsolved", unsolved, torch.int8, (rows, cols), chunk.device, dense=True)
    workspace = _workspace("pits", rows, cols, chunk.device, workspace)
    info = (ctypes.c_int64 * 3)()
    _native.check(
        _native.lib().ofl_breach_single_cell_pits_f32(
            chunk.data_ptr(), rows, cols, chunk.stride(0), float(nodata_value), unsolved.data_ptr(), info,
            workspace.data_ptr(), workspace.numel(), _native.OFL_MEM_DEVICE, _stream(chunk),
        )
    )
    return unsolved, [int(v) for v in info]


# ---------------------------------------------------------------- row strips (strips.py)
# These calls run several times per multi-GPU step and only enqueue work, so they make no Python checks: the library
# checks their sizes, pointers, pitches and workspaces before it touches the device.  `fdr_halo` is a strip's codes
# with one halo row above and below; `record` is its boundary record block (strips.record_bytes).
def strip_workspace(rows, cols, device="cuda") -> torch.Tensor:
    return _workspace("strip", rows, cols, device)


def strip_boundary_workspace(n_strips, cols, device="cuda") -> torch.Tensor:
    return _workspace("strip_boundary", n_strips, cols, device)


def strip_accum_local(fdr_halo, has_above, has_below, fac, workspace, record):
    """Strip-local counts into `fac` and the strip's boundary record into `record` (ofl_strip_accum_local)."""
    _init_for(fac)
    rows, cols = fac.shape
    _native.check(_native.lib().ofl_strip_accum_local(
        fdr_halo.data_ptr(), rows, cols, fdr_halo.stride(0), int(has_above), int(has_below), fac.data_ptr(),
        fac.stride(0), workspace.data_ptr(), workspace.numel(), record.data_ptr(), _stream(fac)))


def strip_boundary_solve(records_all, cols, J_all, workspace):
    """Inflow J_all [n_strips, 2, cols] of every strip's boundary cells from the gathered records
    [n_strips, record bytes] (ofl_strip_boundary_solve)."""
    _init_for(J_all)
    _native.check(_native.lib().ofl_strip_boundary_solve(
        records_all.data_ptr(), records_all.shape[0], cols, J_all.data_ptr(), workspace.data_ptr(), workspace.numel(),
        _stream(J_all)))


def strip_accum_final(fdr_halo, has_above, has_below, J_mine, workspace, fac):
    """The strip's final counts into `fac`: its inflow J_mine [2, cols] pushed down the strip (ofl_strip_accum_final)."""
    _init_for(fac)
    rows, cols = fac.shape
    _native.check(_native.lib().ofl_strip_accum_final(
        fdr_halo.data_ptr(), rows, cols, fdr_halo.stride(0), int(has_above), int(has_below), J_mine.data_ptr(),
        workspace.data_ptr(), workspace.numel(), fac.data_ptr(), fac.stride(0), _stream(fac)))


def strip_collect_flags(workspace, rows, cols, boundary_workspace, n_strips, out):
    """Error flags of the strip calls since the last strip_accum_local (and of the boundary solve) into the int32[4]
    tensor `out`; either workspace may be None.  Stream-ordered, no synchronisation (ofl_strip_collect_flags)."""
    _init_for(out)
    _native.check(_native.lib().ofl_strip_collect_flags(
        workspace.data_ptr() if workspace is not None else None, rows, cols,
        boundary_workspace.data_ptr() if boundary_workspace is not None else None, n_strips, out.data_ptr(),
        _stream(out)))


def strip_check_accumulation(fdr_halo, fac, fac_above, fac_below) -> int:
    """Cells of the strip violating the accumulation recurrence, its first and last rows checked against the
    neighbouring strips' boundary counts fac_above / fac_below (None at the raster's edge); synchronises the stream
    (ofl_strip_check_accumulation_u8)."""
    _init_for(fac)
    rows, cols = fac.shape
    n_bad = ctypes.c_int64(0)
    _native.check(_native.lib().ofl_strip_check_accumulation_u8(
        fdr_halo.data_ptr(), rows, cols, fdr_halo.stride(0), fac.data_ptr(), fac.stride(0),
        fac_above.data_ptr() if fac_above is not None else None,
        fac_below.data_ptr() if fac_below is not None else None, ctypes.byref(n_bad), _stream(fac)))
    return int(n_bad.value)
