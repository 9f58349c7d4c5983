"""Flat resolution -- host-side mirror of the reference's src/overflow/fix_flats.py (Barnes, Lehman & Mulla 2014).

Same names, arguments and results as the reference: `flat_edges` (:13-62), `label_flats` (:65-108),
`away_from_higher` (:111-161), `towards_lower` (:164-224), `resolve_flats` (:227-288) and
`d8_masked_flow_dirs` (:291-339).  The compute is csrc/flats.cu behind the C ABI (ofl_flat_edges_f32,
ofl_resolve_flats_f32, ofl_flat_gradient_i32, ofl_d8_masked_flow_dirs_i32, ofl_fix_flats_f32); there is
no CPU fallback.  `fix_flats_for_tile` chains resolve_flats and d8_masked_flow_dirs in one library call.

Elevations are compared (==, <) in float32 on the device: float32 DEMs are used as they are, other dtypes
are accepted when every value is exactly representable in float32 (which keeps both comparisons
unchanged) and rejected otherwise.
"""
import ctypes

import numpy as np

from . import _native
from .constants import FLOW_DIRECTION_UNDEFINED
from .flow_accumulation import as_codes

_MAX_CELLS = 2**32


def _dem_f32(dem) -> np.ndarray:
    dem = np.asarray(dem)
    if dem.ndim != 2:
        raise ValueError("dem must be a 2-D array")
    if dem.dtype != np.float32:
        as32 = dem.astype(np.float32)
        same = (as32.astype(dem.dtype) == dem) | ((dem != dem) & (as32 != as32))
        if not bool(np.all(same)):
            raise TypeError(f"{dem.dtype} elevations that float32 cannot hold exactly are not supported")
        dem = as32
    return np.ascontiguousarray(dem)


def _codes(fdr, like) -> np.ndarray:
    fdr = as_codes(fdr)
    if fdr.shape != like.shape:
        raise ValueError(f"shape mismatch: {fdr.shape} vs {like.shape}")
    return fdr


def _i32(a, what, like) -> np.ndarray:
    a = np.asarray(a)
    if a.shape != like.shape:
        raise ValueError(f"{what}: shape {a.shape} does not match {like.shape}")
    if a.dtype != np.int32:
        if not np.issubdtype(a.dtype, np.integer):
            raise TypeError(f"{what} must be an integer array, got {a.dtype}")
        if a.size and (a.min() < -(2**31) or a.max() > 2**31 - 1):
            raise ValueError(f"{what} does not fit int32")
        a = a.astype(np.int32)
    return np.ascontiguousarray(a)


def _check_size(shape):
    if shape[0] * shape[1] > _MAX_CELLS:
        raise ValueError("flat resolution works on one tile of at most 2**32 cells")


def flat_edges(dem: np.ndarray, fdr: np.ndarray):
    """(high_edges, low_edges): lists of (row, col) in row-major order (reference :13-62)."""
    dem = _dem_f32(dem)
    fdr = _codes(fdr, dem)
    _check_size(dem.shape)
    rows, cols = dem.shape
    edges = np.zeros((rows, cols), dtype=np.uint8)
    n_low, n_high = ctypes.c_int64(0), ctypes.c_int64(0)
    _native.check(
        _native.lib().ofl_flat_edges_f32(
            dem.ctypes.data, fdr.ctypes.data, rows, cols, edges.ctypes.data, ctypes.byref(n_low), ctypes.byref(n_high),
            _native.OFL_MEM_HOST, None,
        )
    )
    high = [(int(r), int(c)) for r, c in zip(*np.nonzero(edges & 2))]
    low = [(int(r), int(c)) for r, c in zip(*np.nonzero(edges & 1))]
    assert len(low) == n_low.value and len(high) == n_high.value
    return high, low


def resolve_flats(dem: np.ndarray, flow_dirs: np.ndarray, return_info: bool = False):
    """(flat_mask int32, labels int32) of one tile (reference :227-288).

    With return_info also a dict: low / high edge counts, label count, BFS levels of the two sweeps.
    """
    dem = _dem_f32(dem)
    fdr = _codes(flow_dirs, dem)
    _check_size(dem.shape)
    rows, cols = dem.shape
    flat_mask = np.zeros((rows, cols), dtype=np.int32)
    labels = np.zeros((rows, cols), dtype=np.int32)
    info = (ctypes.c_int64 * 5)()
    _native.check(
        _native.lib().ofl_resolve_flats_f32(
            dem.ctypes.data, fdr.ctypes.data, rows, cols, flat_mask.ctypes.data, labels.ctypes.data, info, None, 0,
            _native.OFL_MEM_HOST, None,
        )
    )
    if return_info:
        keys = ("low_edges", "high_edges", "labels", "away_levels", "towards_levels")
        return flat_mask, labels, dict(zip(keys, (int(v) for v in info)))
    return flat_mask, labels


def d8_masked_flow_dirs(flat_mask: np.ndarray, fdr: np.ndarray, labels: np.ndarray) -> None:
    """Give every cell without a direction the direction of its lowest-mask neighbour in the same flat,
    in place (reference :291-339)."""
    if not isinstance(fdr, np.ndarray) or fdr.dtype != np.uint8 or fdr.ndim != 2:
        raise TypeError("fdr must be a 2-D uint8 numpy array (it is modified in place)")
    _check_size(fdr.shape)
    fm = _i32(flat_mask, "flat_mask", fdr)
    lb = _i32(labels, "labels", fdr)
    work = fdr if fdr.flags.c_contiguous else np.ascontiguousarray(fdr)
    rows, cols = work.shape
    _native.check(
        _native.lib().ofl_d8_masked_flow_dirs_i32(
            fm.ctypes.data, lb.ctypes.data, work.ctypes.data, rows, cols, _native.OFL_MEM_HOST, None
        )
    )
    if work is not fdr:
        fdr[...] = work


def _gradient(labels, flat_mask, fdr, edge_list, flat_height, towards):
    if not isinstance(flat_mask, np.ndarray) or flat_mask.ndim != 2 or not np.issubdtype(flat_mask.dtype, np.integer):
        raise TypeError("flat_mask must be a 2-D integer numpy array (it is modified in place)")
    fdr = _codes(fdr, flat_mask)
    _check_size(fdr.shape)
    lb = _i32(labels, "labels", flat_mask)
    fm = _i32(flat_mask, "flat_mask", flat_mask).copy()
    rows, cols = fm.shape
    fh_in = np.asarray(flat_height)
    fh = np.ascontiguousarray(fh_in, dtype=np.int32).copy()
    cells = [(int(r), int(c)) for r, c in edge_list if not (r == -1 and c == -1)]
    for r, c in cells:
        if not (0 <= r < rows and 0 <= c < cols):
            raise IndexError(f"edge cell ({r}, {c}) outside the {rows}x{cols} raster")
    seeds = np.asarray([r * cols + c for r, c in cells], dtype=np.int32)
    if len(seeds) and (lb.ravel()[seeds].max() > len(fh) or (not towards and lb.ravel()[seeds].min() < 1)):
        raise IndexError("a seed cell's label has no flat_height entry")
    _native.check(
        _native.lib().ofl_flat_gradient_i32(
            lb.ctypes.data, fdr.ctypes.data, rows, cols, seeds.ctypes.data if len(seeds) else None, len(seeds),
            1 if towards else 0, fm.ctypes.data, fh.ctypes.data if len(fh) else None, len(fh), None, 0,
            _native.OFL_MEM_HOST, None,
        )
    )
    flat_mask[...] = fm
    if not towards and isinstance(flat_height, np.ndarray):
        flat_height[...] = fh


def away_from_higher(labels, flat_mask, fdr, high_edges, flat_height) -> None:
    """Gradient away from higher terrain: flat_mask and flat_height are filled in place (reference :111-161)."""
    _gradient(labels, flat_mask, fdr, high_edges, flat_height, towards=False)


def towards_lower(labels, flat_mask, fdr, low_edges, flat_height) -> None:
    """Gradient towards lower terrain combined with the one away from higher terrain, in place (:164-224)."""
    _gradient(labels, flat_mask, fdr, low_edges, flat_height, towards=True)


def label_flats(dem, labels, new_label, flat_row, flat_col) -> None:
    """Give the flat containing (flat_row, flat_col) -- every cell reachable over cells of that elevation,
    8-connected -- the label `new_label`, in place, leaving already labelled cells alone (reference :65-108).

    The device labels ALL flats of a tile at once (resolve_flats); this single-flat entry point runs the same
    equal-elevation component search there by resolving a tile in which the start cell is the only low edge.
    """
    dem = _dem_f32(dem)
    if not isinstance(labels, np.ndarray) or labels.shape != dem.shape:
        raise ValueError("labels must be a numpy array of the DEM's shape")
    rows, cols = dem.shape
    if not (0 <= flat_row < rows and 0 <= flat_col < cols):
        return  # the reference pops the start cell, finds it out of bounds and stops
    # Codes under which the start cell is the tile's only possible low edge: it alone "has a direction".  It
    # is a low edge iff a neighbour shares its elevation; resolve_flats then labels exactly its component 1.
    elev = dem[flat_row, flat_col]
    if not (elev == elev):
        return  # NaN never equals itself: the reference labels nothing
    if labels[flat_row, flat_col] != 0:
        return  # the reference pops the start cell, finds it labelled and stops
    # the reference's flood does not pass through cells that already carry a label: they become NaN here, which
    # equals nothing, so the device's equal-elevation components stop at them exactly like the flood does
    taken = labels != 0
    if bool(taken.any()):
        dem = dem.copy()
        dem[taken] = np.nan
    fdr = np.full(dem.shape, FLOW_DIRECTION_UNDEFINED, dtype=np.uint8)
    fdr[flat_row, flat_col] = 0
    r0, r1 = max(0, flat_row - 1), min(rows, flat_row + 2)
    c0, c1 = max(0, flat_col - 1), min(cols, flat_col + 2)
    if int((dem[r0:r1, c0:c1] == elev).sum()) <= 1:
        labels[flat_row, flat_col] = new_label  # a flat of one cell: nothing to search
        return
    _, got = resolve_flats(dem, fdr)
    if got[flat_row, flat_col] == 0:
        raise RuntimeError("label_flats: start cell was not labelled")
    labels[got == got[flat_row, flat_col]] = new_label


def fix_flats_for_tile(dem: np.ndarray, fdr: np.ndarray, return_mask: bool = False):
    """resolve_flats + d8_masked_flow_dirs in one library call (ofl_fix_flats_f32).

    Returns the rewritten codes (a new uint8 array), or (codes, flat_mask, labels) with return_mask.
    """
    dem = _dem_f32(dem)
    out = _codes(fdr, dem).copy()
    _check_size(dem.shape)
    rows, cols = dem.shape
    flat_mask = np.zeros((rows, cols), dtype=np.int32) if return_mask else None
    labels = np.zeros((rows, cols), dtype=np.int32) if return_mask else None
    _native.check(
        _native.lib().ofl_fix_flats_f32(
            dem.ctypes.data, out.ctypes.data, rows, cols, flat_mask.ctypes.data if return_mask else None,
            labels.ctypes.data if return_mask else None, None, None, 0, _native.OFL_MEM_HOST, None,
        )
    )
    return (out, flat_mask, labels) if return_mask else out
