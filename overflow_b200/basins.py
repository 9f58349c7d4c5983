"""Drainage basins: label every cell with the outlet (or pour point) its D8 path reaches.

Uses the accumulation's edge rule: a cell drains into its downstream neighbour when its code is 0..7, the neighbour
lies inside the raster and is not NODATA (9).  A data cell that drains nowhere is an outlet; outlet (r, c) has the
label ``r * cols + c + 1`` and every cell upstream of it gets that label.  NODATA cells get 0.

With pour points -- an ``(k, 2)`` array of ``(row, col)`` -- the call delineates watersheds instead: a pour point
is a root (its outgoing edge is cut), a cell gets ``p + 1`` for the first pour point ``p = row * cols + col`` on its
path (the cell itself included), and a cell whose path meets no pour point gets 0.  Nested pour points therefore
give sub-basins.  ``np.unique(labels, return_inverse=True)`` compacts the labels to 0..B.

The labelling runs in liboverflow_b200 (csrc/basins.cu); there is no CPU fallback.
"""
import ctypes

import numpy as np

from . import _native
from .constants import DEFAULT_CHUNK_SIZE
from .flow_accumulation import as_codes

BASIN_NODATA = 0


def pour_point_indices(pour_points, shape):
    """Row-major cell indices of an ``(k, 2)`` array of ``(row, col)`` pour points (None: no pour points).
    Raises ValueError for a malformed array or a point outside a raster of `shape`."""
    if pour_points is None:
        return None
    pp = np.asarray(pour_points)
    if pp.size == 0:
        pp = pp.reshape(0, 2)
    if pp.ndim != 2 or pp.shape[1] != 2:
        raise ValueError(f"pour points must be a (k, 2) array of (row, col), got shape {pp.shape}")
    if not np.issubdtype(pp.dtype, np.integer):
        raise ValueError(f"pour points must be integers, got {pp.dtype}")
    rows, cols = shape
    pp = pp.astype(np.int64)
    outside = (pp[:, 0] < 0) | (pp[:, 0] >= rows) | (pp[:, 1] < 0) | (pp[:, 1] >= cols)
    if outside.any():
        r, c = pp[np.argmax(outside)]
        raise ValueError(f"pour point ({r}, {c}) lies outside the {rows} x {cols} raster")
    return np.ascontiguousarray(pp[:, 0] * cols + pp[:, 1])


def read_pour_points(path):
    """Pour points from a text file with one ``row,col`` per line (``#`` starts a comment)."""
    pp = np.loadtxt(path, delimiter=",", dtype=np.int64, ndmin=2)
    if pp.size == 0:
        raise ValueError(f"{path} lists no pour points")
    if pp.shape[1] != 2:
        raise ValueError(f"{path}: expected one row,col pair per line")
    return pp


def label_basins(flow_direction, pour_points=None) -> np.ndarray:
    """int64 basin label of every cell of a flow-direction raster (see the module docstring)."""
    fdr = as_codes(flow_direction)
    idx = pour_point_indices(pour_points, fdr.shape)
    rows, cols = fdr.shape
    labels = np.empty((rows, cols), dtype=np.int64)
    n_pour = 0 if idx is None else len(idx)
    if rows and cols:
        _native.check(
            _native.lib().ofl_label_basins_u8(
                fdr.ctypes.data, rows, cols, cols, idx.ctypes.data if n_pour else None, n_pour, labels.ctypes.data,
                cols, None, 0, _native.OFL_MEM_HOST, None,
            )
        )
    return labels


def check_basins(flow_direction, labels, pour_points=None) -> int:
    """Cells that break the labelling rule; 0 proves `labels` exact on an acyclic raster."""
    fdr = as_codes(flow_direction)
    labels = np.ascontiguousarray(labels, dtype=np.int64)
    if labels.shape != fdr.shape:
        raise ValueError("labels must have the flow-direction raster's shape")
    idx = pour_point_indices(pour_points, fdr.shape)
    rows, cols = fdr.shape
    n_pour = 0 if idx is None else len(idx)
    n_bad = ctypes.c_int64(0)
    _native.check(
        _native.lib().ofl_check_basins_u8(
            fdr.ctypes.data, rows, cols, cols, idx.ctypes.data if n_pour else None, n_pour, labels.ctypes.data, cols,
            ctypes.byref(n_bad), _native.OFL_MEM_HOST, None,
        )
    )
    return int(n_bad.value)


def basins(input_path, output_path, chunk_size=DEFAULT_CHUNK_SIZE, pour_points=None):
    """Basin-label GeoTIFF from a flow-direction GeoTIFF: band 1 in, a 1-band Int64 GeoTIFF with nodata 0 and the
    input's projection and geotransform out.  The raster is read whole and labelled in one library call;
    `chunk_size` is the number of rows read and written at a time."""
    from .util import raster as _raster

    src = _raster.open_raster(input_path)
    fdr = _raster.read_band(src.GetRasterBand(1), chunk_size)
    labels = label_basins(fdr, pour_points)
    dst = _raster.create_raster(
        output_path, src.RasterXSize, src.RasterYSize, "Int64",
        projection=src.GetProjection(), geotransform=src.GetGeoTransform(),
    )
    out_band = dst.GetRasterBand(1)
    out_band.SetNoDataValue(BASIN_NODATA)
    _raster.write_band(out_band, labels, chunk_size)
    dst.FlushCache()
    dst = None
