"""D8 flow direction -- host-side mirror of the reference's src/overflow/flow_direction.py.

`flow_direction_for_tile` (reference :14-69) and `flow_direction` (reference :99-124) keep
their signatures; the stencil runs in liboverflow_b200 (csrc/direction.cu).
"""
import ctypes

import numpy as np

from . import _native
from .constants import FLOW_DIRECTION_NODATA

def _classify(dem: np.ndarray):
    """(kind, array) for the C ABI.  kind None: the float32 TMA kernel; otherwise an ofl_elem_kind for
    ofl_flow_direction_x64.  The reference's arithmetic follows the array dtype under numba
    (flow_direction.py:94-96): float32 differences for float32, float64 for float64, int64 for signed
    integers and uint64 -- wrapping for uphill neighbours -- for unsigned ones.  int8/int16 differences
    are exact in float32, so those share the float32 kernel."""
    dt = dem.dtype
    if dt == np.float32:
        return None, dem
    if dt in (np.dtype(np.int8), np.dtype(np.int16)):
        return None, dem.astype(np.float32)
    if dt == np.float64:
        return _native.OFL_ELEM_F64, dem
    if np.issubdtype(dt, np.signedinteger):
        return _native.OFL_ELEM_I64, dem.astype(np.int64)
    if np.issubdtype(dt, np.unsignedinteger):
        return _native.OFL_ELEM_U64, dem.astype(np.uint64)
    raise TypeError(f"flow direction: DEM dtype {dt} is not supported (float32, float64 or an integer type)")


def _as_f32(dem: np.ndarray) -> np.ndarray:
    """float32 view of a DEM that the float32 kernel reproduces exactly, else TypeError."""
    kind, arr = _classify(dem)
    if kind is not None:
        raise TypeError(f"DEM dtype {dem.dtype} does not take the float32 path")
    return arr


def _run_direction(dem, nodata_value, out, mode):
    kind, src = _classify(dem)
    src = np.ascontiguousarray(src)
    rows, cols = src.shape
    lib = _native.lib()
    if kind is None:
        _native.check(lib.ofl_flow_direction_f32(src.ctypes.data, rows, cols, cols, float(nodata_value), out.ctypes.data,
                                                 cols, mode, _native.OFL_MEM_HOST, None))
    else:
        _native.check(lib.ofl_flow_direction_x64(src.ctypes.data, kind, rows, cols, cols, float(nodata_value),
                                                 out.ctypes.data, cols, mode, _native.OFL_MEM_HOST, None))


def _stream_ptr(stream):
    return ctypes.c_void_p(int(stream)) if stream else None


def flow_direction_for_tile(dem: np.ndarray, nodata_value: float) -> np.ndarray:
    """D8 codes for the interior of a DEM chunk that carries a one-cell ring.

    Same contract as the reference (flow_direction.py:14-69): returns uint8 of dem.shape;
    interior cells hold E=0..SE=7, 8 (no downhill neighbour) or 9 (nodata).  The ring, which
    the reference leaves uninitialised, is set to 9.
    """
    dem = np.asarray(dem)
    if dem.ndim != 2:
        raise ValueError("dem must be a 2-D array")
    _classify(dem)  # unsupported dtypes raise before anything is allocated
    rows, cols = dem.shape
    out = np.empty((rows, cols), dtype=np.uint8)
    if rows == 0 or cols == 0:
        return out
    _run_direction(dem, nodata_value, out, _native.OFL_DIR_MODE_TILE)
    return out


def flow_direction_for_raster(dem: np.ndarray, nodata_value: float, out: np.ndarray = None) -> np.ndarray:
    """Whole-raster D8 codes: every cell computed, out-of-raster neighbours read as nodata.

    Equals what `flow_direction()` writes for the file (the chunk loop pads the raster edge
    with the band nodata value, util/raster.py:67); no ring is needed or returned.  `out` may be
    a preallocated C-contiguous uint8 array (e.g. pinned memory) of dem.shape.
    """
    dem = np.asarray(dem)
    if dem.ndim != 2:
        raise ValueError("dem must be a 2-D array")
    _classify(dem)
    rows, cols = dem.shape
    if out is None:
        out = np.empty((rows, cols), dtype=np.uint8)
    elif out.dtype != np.uint8 or out.shape != (rows, cols) or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous uint8 array of dem.shape")
    if rows == 0 or cols == 0:
        return out
    _run_direction(dem, nodata_value, out, _native.OFL_DIR_MODE_RASTER)
    return out


def flow_direction(input_path, output_path, chunk_size=4000):
    """Generate a flow-direction GeoTIFF from a DEM file (reference flow_direction.py:99-124).

    Band 1 of `input_path` is read; the output is a 1-band Byte GeoTIFF with the same
    projection / geotransform and nodata 9.  `chunk_size` keeps its meaning as the I/O
    granularity; the result does not depend on it.  Float32 DEMs go through the band pipeline of
    streaming.py (file reads, PCIe copies, the stencil and file writes overlapped, rows streamed in bands of
    chunk_size rows); every other band type, which needs the generic stencil, and an empty raster take the
    reference's own chunk loop, one synchronous library call per chunk.
    """
    from .util import raster as _raster

    src = _raster.open_raster(input_path)
    band = src.GetRasterBand(1)
    nodata_value = band.GetNoDataValue()
    if _raster.gdal_data_type_to_numpy_data_type(band.DataType) == np.float32 and band.XSize * band.YSize > 0:
        from .streaming import stream_routing

        src = band = None
        stream_routing(input_path, output_path, None, band_rows=chunk_size)
        return
    dst = _raster.create_raster(
        output_path, src.RasterXSize, src.RasterYSize, "Byte",
        projection=src.GetProjection(), geotransform=src.GetGeoTransform(),
    )
    out_band = dst.GetRasterBand(1)
    out_band.SetNoDataValue(FLOW_DIRECTION_NODATA)
    for chunk in _raster.raster_chunker(band, chunk_size=chunk_size, chunk_buffer_size=1):
        result = flow_direction_for_tile(chunk.data, nodata_value)
        chunk.from_numpy(result)
        chunk.write(out_band)
    dst.FlushCache()
    dst = None
