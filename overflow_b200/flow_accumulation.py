"""D8 flow accumulation -- host-side mirror of the reference's src/overflow/flow_accumulation.py.

`single_tile_flow_accumulation` (reference :95-158) keeps its signature and result; counts
and perimeter links come from liboverflow_b200 (csrc/accumulation.cu).  `get_next_cell`,
`perimeter_indices` and `follow_path` are the reference's scalar helpers (:13-92), kept
importable with the same behaviour; they are plain host utilities, not the compute path.
"""
import numpy as np

from . import _native
from .constants import (
    FLOW_DIRECTION_NODATA,
    FLOW_DIRECTION_UNDEFINED,
    FLOW_ACCUMULATION_NODATA,
    FLOW_EXTERNAL,
    FLOW_TERMINATES,
    NEIGHBOR_OFFSETS,
)


def get_next_cell(flow_direction: np.ndarray, row: int, col: int):
    """(row, col, value) of the downstream cell (reference :13-37).

    Codes 8/9 have no offset; the reference's out-of-bounds table read lands "outside the
    tile", so the value is NODATA and the coordinates are not meaningful (returned as -1,-1).
    """
    value = int(flow_direction[row, col])
    if value < 0 or value >= 8:
        return -1, -1, FLOW_DIRECTION_NODATA
    d_row, d_col = NEIGHBOR_OFFSETS[value]
    next_row, next_col = row + int(d_row), col + int(d_col)
    rows, cols = flow_direction.shape
    if 0 <= next_row < rows and 0 <= next_col < cols:
        return next_row, next_col, int(flow_direction[next_row, next_col])
    return next_row, next_col, FLOW_DIRECTION_NODATA


def perimeter_indices(shape):
    """Perimeter (row, col) list in the reference's order (:40-51)."""
    rows, cols = shape
    indices = []
    for i in range(rows):
        indices.append((i, 0))
        indices.append((i, cols - 1))
    for j in range(1, cols - 1):
        indices.append((0, j))
        indices.append((rows - 1, j))
    return indices


def follow_path(flow_direction, row, col, links):
    """Walk downstream from a perimeter cell and record where it leaves the tile (:54-92)."""
    init_row, init_col = row, col
    rows, cols = flow_direction.shape
    for _ in range(rows * cols + 1):
        next_row, next_col, next_val = get_next_cell(flow_direction, row, col)
        inside = 0 <= next_row < rows and 0 <= next_col < cols
        if not inside:
            if row == init_row and col == init_col:
                links[init_row, init_col] = FLOW_EXTERNAL
            else:
                links[init_row, init_col] = (row, col)
            return
        if next_val in (FLOW_DIRECTION_NODATA, FLOW_DIRECTION_UNDEFINED):
            links[init_row, init_col] = FLOW_TERMINATES
            return
        row, col = next_row, next_col
    raise ValueError("flow direction raster contains a cycle")


def as_codes(flow_direction) -> np.ndarray:
    """A flow-direction raster as the C-contiguous uint8 codes the library takes.  Any integer dtype is accepted;
    a code outside 0..255 raises ValueError instead of wrapping."""
    fdr = np.asarray(flow_direction)
    if fdr.ndim != 2:
        raise ValueError("flow direction raster must be a 2-D array")
    if fdr.dtype != np.uint8:
        if not np.issubdtype(fdr.dtype, np.integer):
            raise TypeError(f"flow direction codes must be integers, got {fdr.dtype}")
        if fdr.size and (fdr.min() < 0 or fdr.max() > 255):
            raise ValueError("flow direction codes must be in 0..255")
        fdr = fdr.astype(np.uint8)
    return np.ascontiguousarray(fdr)


def flow_accumulation_for_raster(flow_direction: np.ndarray, with_links: bool = False, out: np.ndarray = None):
    """int64 upstream-cell counts for a whole flow-direction raster (+ perimeter links).

    Returns fac, or (fac, perim_links[n,2]) with the links in perimeter_indices order.
    NODATA cells hold -9998 exactly as the reference leaves them.  `out` may be a preallocated
    C-contiguous int64 array (e.g. pinned memory) of the raster's shape.
    """
    fdr = as_codes(flow_direction)
    rows, cols = fdr.shape
    if out is None:
        fac = np.empty((rows, cols), dtype=np.int64)
    elif out.dtype != np.int64 or out.shape != (rows, cols) or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous int64 array of the raster's shape")
    else:
        fac = out
    lib = _native.lib()
    n_perim = int(lib.ofl_perimeter_count(rows, cols))
    perim = np.empty((n_perim, 2), dtype=np.int64) if with_links else None
    if rows and cols:
        _native.check(
            lib.ofl_flow_accumulation_u8(
                fdr.ctypes.data, rows, cols, cols, fac.ctypes.data, cols,
                perim.ctypes.data if with_links else None, None, 0, _native.OFL_MEM_HOST, None,
            )
        )
    return (fac, perim) if with_links else fac


def single_tile_flow_accumulation(flow_direction: np.ndarray):
    """Flow accumulation and perimeter links of one tile (reference :95-158).

    Returns (flow_accumulation int64[R,C], links int64[R,C,2]).  Perimeter entries of `links`
    are FLOW_EXTERNAL / FLOW_TERMINATES / the (row, col) of the exit cell; interior entries,
    uninitialised in the reference, are zero.
    """
    fdr = as_codes(flow_direction)
    fac, perim = flow_accumulation_for_raster(fdr, with_links=True)
    links = np.zeros(fdr.shape + (2,), dtype=np.int64)
    if len(perim):
        idx = np.asarray(perimeter_indices(fdr.shape), dtype=np.int64).reshape(-1, 2)
        links[idx[:, 0], idx[:, 1]] = perim
    return fac, links


def check_flow_accumulation(flow_direction: np.ndarray, flow_accumulation_raster: np.ndarray) -> int:
    """Cells violating fac = 1 + sum(upstream fac) (data) or fac = -9998 (nodata); 0 proves exactness."""
    import ctypes

    fdr = as_codes(flow_direction)
    fac = np.ascontiguousarray(flow_accumulation_raster, dtype=np.int64)
    rows, cols = fdr.shape
    n_bad = ctypes.c_int64(0)
    _native.check(
        _native.lib().ofl_check_accumulation_u8(
            fdr.ctypes.data, rows, cols, cols, fac.ctypes.data, cols, ctypes.byref(n_bad), _native.OFL_MEM_HOST, None
        )
    )
    return int(n_bad.value)


def flow_accumulation(input_path, output_path, chunk_size=2000):
    """Flow-accumulation GeoTIFF from a flow-direction GeoTIFF.

    Absent from the reference snapshot (SURVEY.md fact 1); follows the house pattern of
    flow_direction() (flow_direction.py:99-124): band 1 in, 1-band Int64 GeoTIFF out with the
    same projection / geotransform and nodata FLOW_ACCUMULATION_NODATA.  The whole raster is
    accumulated on the device; `chunk_size` is the I/O granularity: the codes go up and the counts come down in
    bands of rows while the files are read and written (streaming.py; an empty raster is read whole, one library
    call, written whole).  NODATA cells hold -9998 in the output, as in the reference's array
    result (SURVEY fact 2), although the band's nodata value is -9999: see INTEGRATION.md section 3.
    """
    from .util import raster as _raster

    src = _raster.open_raster(input_path)
    if src.RasterXSize * src.RasterYSize > 0:
        from .streaming import stream_accumulation

        src = None
        stream_accumulation(input_path, output_path, band_rows=chunk_size)
        return
    band = src.GetRasterBand(1)
    fdr = _raster.read_band(band, chunk_size)
    fac = flow_accumulation_for_raster(fdr)
    dst = _raster.create_raster(
        output_path, src.RasterXSize, src.RasterYSize, "Int64",
        projection=src.GetProjection(), geotransform=src.GetGeoTransform(),
    )
    out_band = dst.GetRasterBand(1)
    out_band.SetNoDataValue(FLOW_ACCUMULATION_NODATA)
    _raster.write_band(out_band, fac, chunk_size)
    dst.FlushCache()
    dst = None
