"""Flow direction followed by flow accumulation in one call.

The reference runs the two steps as separate file-level passes (flow_direction.py:99-124 writes the
codes, a later pass reads them back).  On the GPU the codes can stay in HBM between the two kernels, and
for host rasters the upload of the DEM, the stencil and the download of the codes overlap in row bands
(`ofl_flow_routing_f32`, csrc/api.cu).  Results are identical to `flow_direction_for_raster` followed by
`flow_accumulation_for_raster`.
"""
import numpy as np

from . import _native
from .flow_direction import _classify, flow_direction_for_raster


def flow_routing_for_raster(dem: np.ndarray, nodata_value: float, out_fdr: np.ndarray = None,
                            out_fac: np.ndarray = None, with_links: bool = False, want_fdr: bool = True):
    """(fdr uint8, fac int64[, perim_links]) of a whole DEM held in host memory.

    `out_fdr` / `out_fac` may be preallocated C-contiguous arrays (e.g. pinned memory) of dem.shape.
    With `want_fdr=False` the codes are not copied back and None is returned in their place.
    """
    dem = np.asarray(dem)
    if dem.ndim != 2:
        raise ValueError("dem must be a 2-D array")
    kind, src = _classify(dem)
    if kind is not None:
        # float64 / integer DEMs: the generic stencil, then accumulation of its codes
        from .flow_accumulation import flow_accumulation_for_raster

        fdr = flow_direction_for_raster(dem, nodata_value, out=out_fdr)
        res = flow_accumulation_for_raster(fdr, with_links=with_links, out=out_fac)
        fdr = fdr if want_fdr else None
        return (fdr, res[0], res[1]) if with_links else (fdr, res)
    src = np.ascontiguousarray(src)
    rows, cols = src.shape
    if want_fdr:
        if out_fdr is None:
            out_fdr = np.empty((rows, cols), dtype=np.uint8)
        elif out_fdr.dtype != np.uint8 or out_fdr.shape != (rows, cols) or not out_fdr.flags.c_contiguous:
            raise ValueError("out_fdr must be a C-contiguous uint8 array of dem.shape")
    else:
        out_fdr = None
    if out_fac is None:
        out_fac = np.empty((rows, cols), dtype=np.int64)
    elif out_fac.dtype != np.int64 or out_fac.shape != (rows, cols) or not out_fac.flags.c_contiguous:
        raise ValueError("out_fac must be a C-contiguous int64 array of dem.shape")
    lib = _native.lib()
    perim = np.empty((int(lib.ofl_perimeter_count(rows, cols)), 2), dtype=np.int64) if with_links else None
    if rows and cols:
        _native.check(
            lib.ofl_flow_routing_f32(
                src.ctypes.data, rows, cols, cols, float(nodata_value),
                out_fdr.ctypes.data if want_fdr else None, cols, out_fac.ctypes.data, cols,
                perim.ctypes.data if with_links else None, _native.OFL_MEM_HOST, None,
            )
        )
    return (out_fdr, out_fac, perim) if with_links else (out_fdr, out_fac)


def flow_routing(input_path, flow_direction_path, flow_accumulation_path, chunk_size=2000):
    """DEM file -> flow-direction GeoTIFF and flow-accumulation GeoTIFF in one pass over the device.

    File-level counterpart of `flow_routing_for_raster`, in the pattern of the reference's
    `flow_direction()` (flow_direction.py:99-124): band 1 in; a 1-band Byte raster (nodata 9) and a 1-band
    Int64 raster (nodata FLOW_ACCUMULATION_NODATA) out, same projection / geotransform.  The outputs equal
    what `flow_direction()` followed by `flow_accumulation()` write; `chunk_size` is the I/O granularity: Float32
    DEMs move through the band pipeline of streaming.py in bands of chunk_size rows (reads, copies, kernels and
    writes overlapped); other band types, whose generic stencil the pipeline lacks, and empty rasters are read
    whole first.
    """
    from .constants import FLOW_ACCUMULATION_NODATA, FLOW_DIRECTION_NODATA
    from .util import raster as _raster

    src = _raster.open_raster(input_path)
    band = src.GetRasterBand(1)
    nodata_value = band.GetNoDataValue()
    assert nodata_value is not None, "the DEM band needs a nodata value (util/raster.py:59 in the reference)"
    if _raster.gdal_data_type_to_numpy_data_type(band.DataType) == np.float32 and band.XSize * band.YSize > 0:
        from .streaming import stream_routing

        src = band = None
        return stream_routing(input_path, flow_direction_path, flow_accumulation_path, band_rows=chunk_size)
    dem = _raster.read_band(band, chunk_size)
    fdr, fac = flow_routing_for_raster(dem, nodata_value)
    for path, name, nodata, arr in ((flow_direction_path, "Byte", FLOW_DIRECTION_NODATA, fdr),
                                    (flow_accumulation_path, "Int64", FLOW_ACCUMULATION_NODATA, fac)):
        dst = _raster.create_raster(path, src.RasterXSize, src.RasterYSize, name, projection=src.GetProjection(),
                                    geotransform=src.GetGeoTransform())
        out_band = dst.GetRasterBand(1)
        out_band.SetNoDataValue(nodata)
        _raster.write_band(out_band, arr, chunk_size)
        dst.FlushCache()
        dst = None
