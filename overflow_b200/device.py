"""Device-resident entry points: torch CUDA tensors in, torch CUDA tensors out.

PyTorch is only the owner of device memory and streams here; every kernel is in
liboverflow_b200.  Calls are enqueued on torch's current stream.
"""
import ctypes

import torch

from . import _native


def _stream(t=None):
    """torch's current stream on the tensor's device (not on whatever device happens to be current)."""
    return ctypes.c_void_p(torch.cuda.current_stream(t.device if t is not None else None).cuda_stream)


def _init_for(t: torch.Tensor):
    if not t.is_cuda:
        raise ValueError("expected a CUDA tensor (there is no CPU fallback)")
    _native.init(t.device.index if t.device.index is not None else torch.cuda.current_device())


def _pitched(rows, cols, dtype, device, align):
    """rows x cols view of a buffer whose row pitch is a multiple of `align` elements (the library's TMA tensor
    maps want 16-byte pitches; a dense tensor of odd width does not have one)."""
    return torch.empty((rows, (cols + align - 1) // align * align), dtype=dtype, device=device)[:, :cols]


def _check_raster(name, t, dtype, shape, like, pitch_align=1):
    """Raw pointers of `t` go straight into the C ABI: refuse anything it would mis-read."""
    if not isinstance(t, torch.Tensor) or t.dtype != dtype or t.dim() != 2 or tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} must be a {dtype} tensor of shape {tuple(shape)}")
    if t.device != like.device:
        raise ValueError(f"{name} must live on {like.device}, not {t.device}")
    if t.shape[1] > 1 and t.stride(1) != 1:
        raise ValueError(f"{name} must have unit column stride")
    if t.shape[0] > 1 and (t.stride(0) < t.shape[1] or t.stride(0) % pitch_align):
        raise ValueError(f"{name}: row pitch {t.stride(0)} must be >= {t.shape[1]} and a multiple of {pitch_align}")
    return t


def _check_workspace(name, t, need, like):
    if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or t.dim() != 1 or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous 1-D uint8 tensor")
    if t.device != like.device:
        raise ValueError(f"{name} must live on {like.device}, not {t.device}")
    if t.numel() < need:
        raise ValueError(f"{name} holds {t.numel()} bytes, {need} needed")
    return t


def synth_dem(rows, cols, *, row0=0, total_rows=None, seed=0, kind=0, relief=1000.0, holes_permille=0,
              nodata=-9999.0, device="cuda", out=None):
    """Seeded synthetic float32 DEM generated on the device (kind 0 fractal, 1 terraces, 2 tilted plane,
    3 walled serpentine: one channel of about rows * cols / 2 cells running east-west; 4 the same running north-south).

    Rows row0..row0+rows-1 of a raster with `total_rows` rows; rows outside [0,total_rows) are nodata
    (that is what a strip's halo row is at the raster top / bottom).  `out`: write into this tensor.
    """
    total_rows = rows if total_rows is None else total_rows
    if out is None:
        dem = _pitched(rows, cols, torch.float32, device, 4)
    else:
        if not out.is_cuda:
            raise ValueError("expected a CUDA tensor (there is no CPU fallback)")
        dem = _check_raster("out", out, torch.float32, (rows, cols), out)
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
    if dem.dtype != torch.float32 or dem.dim() != 2 or dem.stride(1) != 1:
        raise ValueError("dem must be a 2-D float32 tensor with unit column stride")
    _init_for(dem)
    m = {"tile": _native.OFL_DIR_MODE_TILE, "raster": _native.OFL_DIR_MODE_RASTER, "strip": _native.OFL_DIR_MODE_STRIP}[mode]
    rows, cols = dem.shape
    if m == _native.OFL_DIR_MODE_STRIP:
        rows -= 2
    if dem.shape[0] and dem.shape[1] and (dem.stride(0) % 4 or dem.data_ptr() % 16):
        dem = _pitched(dem.shape[0], cols, torch.float32, dem.device, 4).copy_(dem)  # dense odd widths: re-pitch (TMA)
    if out is None:
        out = _pitched(rows, cols, torch.uint8, dem.device, 16)  # flow_accumulation wants 16-byte pitches
    else:
        _check_raster("out", out, torch.uint8, (rows, cols), dem, 4)
    _native.check(
        _native.lib().ofl_flow_direction_f32(
            dem.data_ptr(), rows, cols, dem.stride(0), float(nodata_value), out.data_ptr(), out.stride(0), m,
            _native.OFL_MEM_DEVICE, _stream(dem),
        )
    )
    return out


def accumulation_workspace(rows, cols, device="cuda") -> torch.Tensor:
    n = int(_native.lib().ofl_accumulation_workspace_bytes(rows, cols))
    return torch.empty((n,), dtype=torch.uint8, device=device)


def flow_accumulation(fdr: torch.Tensor, *, out=None, workspace=None, with_links=False):
    """int64 upstream-cell counts of a uint8 CUDA flow-direction raster.

    Returns fac, or (fac, perim_links[n,2]) in perimeter_indices order when with_links.
    Synchronises the stream (the perimeter-graph solve reports convergence to the host).
    """
    if fdr.dtype != torch.uint8 or fdr.dim() != 2 or fdr.stride(1) != 1:
        raise ValueError("fdr must be a 2-D uint8 tensor with unit column stride")
    _init_for(fdr)
    rows, cols = fdr.shape
    if rows and cols and (fdr.stride(0) % 16 or fdr.data_ptr() % 16):
        fdr = _pitched(rows, cols, torch.uint8, fdr.device, 16).copy_(fdr)  # dense odd widths: re-pitch (TMA)
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.int64, device=fdr.device)
    else:
        _check_raster("out", out, torch.int64, (rows, cols), fdr)
    need = int(_native.lib().ofl_accumulation_workspace_bytes(rows, cols))
    if workspace is None:
        workspace = accumulation_workspace(rows, cols, fdr.device)
    else:
        _check_workspace("workspace", workspace, need, fdr)
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
    if dem.dtype != torch.float32 or dem.dim() != 2 or dem.stride(1) != 1:
        raise ValueError("dem must be a 2-D float32 tensor with unit column stride")
    _init_for(dem)
    rows, cols = dem.shape
    if resolve_flats:
        if not dem.is_contiguous():
            raise ValueError("resolve_flats needs a contiguous DEM")
        if cols % 16:
            raise ValueError("resolve_flats needs a column count that is a multiple of 16 (dense codes, TMA pitch)")
        fdr = flow_direction(dem, nodata_value, out=out_fdr)
        fix_flats(dem, fdr)
        return fdr, flow_accumulation(fdr, out=out_fac)
    if rows and cols and (dem.stride(0) % 4 or dem.data_ptr() % 16):
        dem = _pitched(rows, cols, torch.float32, dem.device, 4).copy_(dem)  # dense odd widths: re-pitch (TMA)
    if out_fdr is None:
        out_fdr = _pitched(rows, cols, torch.uint8, dem.device, 16)
    else:
        _check_raster("out_fdr", out_fdr, torch.uint8, (rows, cols), dem, 16)
    if out_fac is None:
        out_fac = torch.empty((rows, cols), dtype=torch.int64, device=dem.device)
    else:
        _check_raster("out_fac", out_fac, torch.int64, (rows, cols), dem)
    _native.check(
        _native.lib().ofl_flow_routing_f32(
            dem.data_ptr(), rows, cols, dem.stride(0), float(nodata_value), out_fdr.data_ptr(), out_fdr.stride(0),
            out_fac.data_ptr(), out_fac.stride(0), None, _native.OFL_MEM_DEVICE, _stream(dem),
        )
    )
    return out_fdr, out_fac


def check_accumulation(fdr: torch.Tensor, fac: torch.Tensor) -> int:
    """Number of cells violating the accumulation recurrence (0 proves fac exact on an acyclic raster)."""
    if fdr.dtype != torch.uint8 or fdr.dim() != 2 or (fdr.shape[1] > 1 and fdr.stride(1) != 1):
        raise ValueError("fdr must be a 2-D uint8 tensor with unit column stride")
    _init_for(fdr)
    rows, cols = fdr.shape
    _check_raster("fac", fac, torch.int64, (rows, cols), fdr)
    n_bad = ctypes.c_int64(0)
    _native.check(
        _native.lib().ofl_check_accumulation_u8(
            fdr.data_ptr(), rows, cols, fdr.stride(0), fac.data_ptr(), fac.stride(0), ctypes.byref(n_bad),
            _native.OFL_MEM_DEVICE, _stream(fdr),
        )
    )
    return int(n_bad.value)


def basins_workspace(rows, cols, device="cuda") -> torch.Tensor:
    n = int(_native.lib().ofl_basins_workspace_bytes(rows, cols))
    return torch.empty((n,), dtype=torch.uint8, device=device)


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
    if fdr.dtype != torch.uint8 or fdr.dim() != 2 or fdr.stride(1) != 1:
        raise ValueError("fdr must be a 2-D uint8 tensor with unit column stride")
    _init_for(fdr)
    rows, cols = fdr.shape
    idx = _pour_indices(pour_points, fdr)
    if rows and cols and (fdr.stride(0) % 16 or fdr.data_ptr() % 16):
        fdr = _pitched(rows, cols, torch.uint8, fdr.device, 16).copy_(fdr)  # dense odd widths: re-pitch
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.int64, device=fdr.device)
    else:
        _check_raster("out", out, torch.int64, (rows, cols), fdr)
    need = int(_native.lib().ofl_basins_workspace_bytes(rows, cols))
    if workspace is None:
        workspace = basins_workspace(rows, cols, fdr.device)
    else:
        _check_workspace("workspace", workspace, need, fdr)
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
    if fdr.dtype != torch.uint8 or fdr.dim() != 2 or (fdr.shape[1] > 1 and fdr.stride(1) != 1):
        raise ValueError("fdr must be a 2-D uint8 tensor with unit column stride")
    _init_for(fdr)
    rows, cols = fdr.shape
    _check_raster("labels", labels, torch.int64, (rows, cols), fdr)
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
    n = int(_native.lib().ofl_flats_workspace_bytes(rows, cols))
    return torch.empty((max(n, 256),), dtype=torch.uint8, device=device)


def _flats_args(dem, fdr):
    if dem.dtype != torch.float32 or dem.dim() != 2 or not dem.is_contiguous():
        raise ValueError("dem must be a contiguous 2-D float32 tensor")
    if fdr.dtype != torch.uint8 or fdr.shape != dem.shape or not fdr.is_contiguous():
        raise ValueError("fdr must be a contiguous uint8 tensor of the DEM's shape")
    _init_for(dem)


def resolve_flats(dem: torch.Tensor, fdr: torch.Tensor, *, workspace=None):
    """(flat_mask int32, labels int32, info) of a float32 CUDA DEM and its uint8 codes (ofl_resolve_flats_f32).
    info = [low edges, high edges, labels, away levels, towards levels].  Synchronises the stream."""
    _flats_args(dem, fdr)
    rows, cols = dem.shape
    flat_mask = torch.empty((rows, cols), dtype=torch.int32, device=dem.device)
    labels = torch.empty((rows, cols), dtype=torch.int32, device=dem.device)
    if workspace is None:
        workspace = flats_workspace(rows, cols, dem.device)
    else:
        _check_workspace("workspace", workspace, int(_native.lib().ofl_flats_workspace_bytes(rows, cols)), dem)
    info = (ctypes.c_int64 * 5)()
    _native.check(
        _native.lib().ofl_resolve_flats_f32(
            dem.data_ptr(), fdr.data_ptr(), rows, cols, flat_mask.data_ptr(), labels.data_ptr(), info,
            workspace.data_ptr(), workspace.numel(), _native.OFL_MEM_DEVICE, _stream(dem),
        )
    )
    return flat_mask, labels, [int(v) for v in info]


def fix_flats(dem: torch.Tensor, fdr: torch.Tensor, *, workspace=None, flat_mask=None, labels=None):
    """Rewrite the code-8 cells of `fdr` in place (resolve_flats + d8_masked_flow_dirs, ofl_fix_flats_f32).
    Returns (fdr, info).  Synchronises the stream."""
    _flats_args(dem, fdr)
    rows, cols = dem.shape
    if flat_mask is None:
        flat_mask = torch.empty((rows, cols), dtype=torch.int32, device=dem.device)
    elif not flat_mask.is_contiguous():
        raise ValueError("flat_mask must be contiguous")
    else:
        _check_raster("flat_mask", flat_mask, torch.int32, (rows, cols), dem)
    if labels is None:
        labels = torch.empty((rows, cols), dtype=torch.int32, device=dem.device)
    elif not labels.is_contiguous():
        raise ValueError("labels must be contiguous")
    else:
        _check_raster("labels", labels, torch.int32, (rows, cols), dem)
    if workspace is None:
        workspace = flats_workspace(rows, cols, dem.device)
    else:
        _check_workspace("workspace", workspace, int(_native.lib().ofl_flats_workspace_bytes(rows, cols)), dem)
    info = (ctypes.c_int64 * 5)()
    _native.check(
        _native.lib().ofl_fix_flats_f32(
            dem.data_ptr(), fdr.data_ptr(), rows, cols, flat_mask.data_ptr(), labels.data_ptr(), info,
            workspace.data_ptr(), workspace.numel(), _native.OFL_MEM_DEVICE, _stream(dem),
        )
    )
    return fdr, [int(v) for v in info]


def breach_single_cell_pits(chunk: torch.Tensor, nodata_value: float, *, unsolved=None, workspace=None):
    """Breach the single-cell pits of a float32 CUDA chunk in place (ofl_breach_single_cell_pits_f32).
    Returns (unsolved int8 tensor, [pits found, pits left unsolved, rounds]).  Synchronises the stream."""
    if chunk.dtype != torch.float32 or chunk.dim() != 2 or chunk.stride(1) != 1:
        raise ValueError("chunk must be a 2-D float32 tensor with unit column stride")
    _init_for(chunk)
    rows, cols = chunk.shape
    nbytes = int(_native.lib().ofl_pits_workspace_bytes(rows, cols))
    if unsolved is None:
        unsolved = torch.empty((rows, cols), dtype=torch.int8, device=chunk.device)
    elif not unsolved.is_contiguous():
        raise ValueError("unsolved must be contiguous")
    else:
        _check_raster("unsolved", unsolved, torch.int8, (rows, cols), chunk)
    if workspace is None:
        workspace = torch.empty((max(nbytes, 256),), dtype=torch.uint8, device=chunk.device)
    else:
        _check_workspace("workspace", workspace, nbytes, chunk)
    info = (ctypes.c_int64 * 3)()
    _native.check(
        _native.lib().ofl_breach_single_cell_pits_f32(
            chunk.data_ptr(), rows, cols, chunk.stride(0), float(nodata_value), unsolved.data_ptr(), info,
            workspace.data_ptr(), workspace.numel(), _native.OFL_MEM_DEVICE, _stream(chunk),
        )
    )
    return unsolved, [int(v) for v in info]
