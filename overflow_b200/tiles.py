"""Flow accumulation of a raster cut into RECTANGULAR TILES (SURVEY 8f rank 3): Barnes 2016 as the reference lays
it out.

The reference ships the producer half of the tiled algorithm of the paper it cites (arXiv 1608.04431;
src/overflow/flow_accumulation.py:54-158): `single_tile_flow_accumulation` returns, per tile, the tile-local counts
and `links` -- for every perimeter cell, where its flow path leaves the tile.  This module is the rest of it, with the
device as the producer:

  pass 1   every tile on the device on its own: tile-local counts + perimeter links (`ofl_flow_accumulation_u8`);
           only the perimeter (count, code, link per perimeter cell) is kept
  consumer the graph of ALL tiles' perimeter cells on the host (numpy): an exit cell's D8 step lands on a perimeter
           cell of a neighbouring tile (any of the eight neighbours -- paths cross corners); subtree sums over that
           forest by pointer doubling give J, the inflow every perimeter cell receives from outside its tile
  pass 2   every tile again, seeded with its J on all four sides (`ofl_flow_accumulation_seeded_u8`): final counts

Tiles may have any size (they need not be multiples of the device's 64 x 64 work tile) and the raster need not fit
the device or the host: memory is one tile on the device plus ~30 B per perimeter cell on the host.  The result
equals the whole-raster accumulation bit for bit (integer sums).  Full-width strips (strips.py) are the special case
the multi-GPU path uses; this is the general one.
"""
import numpy as np

from . import _native
from .constants import FLOW_DIRECTION_NODATA
from .flow_accumulation import as_codes

_DY = np.array([0, -1, -1, -1, 0, 1, 1, 1], dtype=np.int64)  # E, NE, N, NW, W, SW, S, SE (constants.py:29-40)
_DX = np.array([1, 1, 0, -1, -1, -1, 0, 1], dtype=np.int64)


def perimeter_cells(rows, cols):
    """(r, c) arrays of perimeter_indices(shape) (reference flow_accumulation.py:40-51), vectorised: every row's left
    then right cell, then for columns 1..C-2 the top then the bottom cell."""
    r = np.repeat(np.arange(rows, dtype=np.int64), 2)
    c = np.tile(np.array([0, cols - 1], dtype=np.int64), rows)
    inner = np.arange(1, max(cols - 1, 1), dtype=np.int64)
    r2 = np.tile(np.array([0, rows - 1], dtype=np.int64), len(inner))
    c2 = np.repeat(inner, 2)
    return np.concatenate([r, r2]), np.concatenate([c, c2])


def perimeter_rank(r, c, rows, cols):
    """Index of perimeter cell (r, c) in perimeter_indices order (its first occurrence, for cells listed twice)."""
    r, c = np.asarray(r, dtype=np.int64), np.asarray(c, dtype=np.int64)
    return np.where(c == 0, 2 * r, np.where(c == cols - 1, 2 * r + 1,
                    np.where(r == 0, 2 * rows + 2 * (c - 1), 2 * rows + 2 * (c - 1) + 1)))


class CudaTileEngine:
    """The product engine: one tile per call through the C ABI (host arrays; the library stages them)."""

    def __init__(self, device=None):
        import torch

        if not torch.cuda.is_available():
            raise _native.OverflowB200Error(-100, "no CUDA device: the tiled driver has no CPU fallback")
        _native.init(torch.cuda.current_device() if device is None else torch.device(device).index or 0)

    def accumulate(self, fdr, inflow=None, want_links=True):
        """(fac int64[h, w], links int64[n_perim, 2] or None) of one tile; `inflow` int64[n_perim] or None."""
        fdr = np.ascontiguousarray(fdr, dtype=np.uint8)
        h, w = fdr.shape
        lib = _native.lib()
        fac = np.empty((h, w), dtype=np.int64)
        n = int(lib.ofl_perimeter_count(h, w))
        links = np.empty((n, 2), dtype=np.int64) if want_links else None
        if inflow is not None:
            inflow = np.ascontiguousarray(inflow, dtype=np.int64)
            if inflow.shape != (n,):
                raise ValueError(f"inflow must have {n} entries (perimeter_indices order), got {inflow.shape}")
        _native.check(lib.ofl_flow_accumulation_seeded_u8(
            fdr.ctypes.data, h, w, w, fac.ctypes.data, w, inflow.ctypes.data if inflow is not None else None,
            links.ctypes.data if want_links else None, None, 0, _native.OFL_MEM_HOST, None))
        return fac, links


def tile_grid(rows, cols, tile_rows, tile_cols):
    """[(r0, r1, c0, c1)] row-major."""
    tile_rows, tile_cols = int(tile_rows), int(tile_cols)
    if tile_rows < 1 or tile_cols < 1:
        raise ValueError("tile_rows and tile_cols must be positive")
    return [(r0, min(rows, r0 + tile_rows), c0, min(cols, c0 + tile_cols))
            for r0 in range(0, rows, tile_rows) for c0 in range(0, cols, tile_cols)]


def solve_perimeter_graph(tiles, rows, cols, tile_rows, tile_cols, perim):
    """The consumer: inflow J per perimeter cell of every tile.

    perim[t] = (count int64[n_t], code uint8[n_t], links int64[n_t, 2]) of tile t in perimeter_indices order.
    Returns [J_t int64[n_t]] with the inflow of a cell listed twice carried by its first entry only.
    """
    n_tc = (cols + tile_cols - 1) // tile_cols
    offs = np.zeros(len(tiles) + 1, dtype=np.int64)
    for t, (_, _, _) in enumerate(perim):
        offs[t + 1] = offs[t] + len(perim[t][0])
    m = int(offs[-1])
    base = np.zeros(m, dtype=np.int64)
    parent = np.full(m, -1, dtype=np.int64)
    code_all = np.concatenate([p[1] for p in perim]) if m else np.zeros(0, dtype=np.uint8)

    def node_of(gr, gc):
        """Global perimeter node of raster cells (gr, gc), which lie on their tiles' perimeters."""
        ti, tj = gr // tile_rows, gc // tile_cols
        t = ti * n_tc + tj
        h = np.minimum(tile_rows, rows - ti * tile_rows)
        w = np.minimum(tile_cols, cols - tj * tile_cols)
        return offs[t] + perimeter_rank(gr - ti * tile_rows, gc - tj * tile_cols, h, w)

    for t, (r0, r1, c0, c1) in enumerate(tiles):
        cnt, code, links = perim[t]
        h, w = r1 - r0, c1 - c0
        pr, pc = perimeter_cells(h, w)
        first = perimeter_rank(pr, pc, h, w) == np.arange(len(pr))  # a cell listed twice acts once
        flows = code < 8
        # the cell's own D8 step: does it leave the tile, and onto what?
        cd = np.where(flows, code, 0).astype(np.int64)
        nr, nc = pr + _DY[cd], pc + _DX[cd]
        leaves = flows & ((nr < 0) | (nr >= h) | (nc < 0) | (nc >= w))
        gr, gc = nr + r0, nc + c0
        inside = leaves & (gr >= 0) & (gr < rows) & (gc >= 0) & (gc < cols)
        tgt = np.full(len(pr), -1, dtype=np.int64)
        if inside.any():
            cand = node_of(gr[inside], gc[inside])
            cand[code_all[cand] == FLOW_DIRECTION_NODATA] = -1  # no edge into a NODATA cell (flow_accumulation.py:118-124)
            tgt[inside] = cand
        # what leaves the tile through this cell is its tile-local count ...
        send = first & (tgt >= 0)
        np.add.at(base, tgt[send], cnt[send])
        # ... and the entry cell it lands on is the parent of every perimeter cell whose path exits here.
        # links: (-2, -2) the path leaves at the cell itself, (-1, -1) it ends inside the tile, else the exit cell
        ext = flows & (links[:, 0] == -2)
        term = links[:, 0] == -1
        exit_k = np.where(ext, np.arange(len(pr)), -1)
        via = flows & ~ext & ~term
        if via.any():
            exit_k[via] = perimeter_rank(links[via, 0], links[via, 1], h, w)
        has = first & (exit_k >= 0)
        parent[offs[t] : offs[t + 1]][has] = tgt[exit_k[has]]
    # subtree sums over the forest by pointer doubling: round j adds every node's sum (complete within distance
    # 2^j below it) to its 2^j-th ancestor, then the node jumps; O(log depth) numpy passes, exact integer sums
    J = base.copy()
    ptr = parent.copy()
    for _ in range(72):
        act = np.nonzero(ptr >= 0)[0]
        if len(act) == 0:
            break
        add = J[act]
        anc = ptr[act]
        nxt = ptr[anc]
        np.add.at(J, anc, add)
        ptr[act] = nxt
    else:
        raise _native.OverflowB200Error(_native.OFL_ERR_CYCLE, "flow-direction raster contains a cycle (tile perimeter graph)")
    return [J[offs[t] : offs[t + 1]].copy() for t in range(len(tiles))]


def flow_accumulation_tiled(read_window, write_window, rows, cols, tile_rows, tile_cols, engine=None, device=None):
    """Flow accumulation of a flow-direction raster through rectangular tiles of (at most) tile_rows x tile_cols.

        read_window(r0, r1, c0, c1) -> uint8 array [r1 - r0, c1 - c0] with the codes of that window
        write_window(r0, c0, fac)      receives the final int64 counts of the window starting at (r0, c0)

    Returns the number of tiles.  See the module docstring for the algorithm.
    """
    if engine is None:
        engine = CudaTileEngine(device)
    tiles = tile_grid(rows, cols, tile_rows, tile_cols)

    def load(t):
        r0, r1, c0, c1 = tiles[t]
        block = as_codes(read_window(r0, r1, c0, c1))
        if block.shape != (r1 - r0, c1 - c0):
            raise ValueError(f"read_window{(r0, r1, c0, c1)} returned shape {block.shape}")
        return block

    perim = []
    for t in range(len(tiles)):
        block = load(t)
        fac, links = engine.accumulate(block, None, True)
        pr, pc = perimeter_cells(*block.shape)
        perim.append((fac[pr, pc].copy(), block[pr, pc].copy(), links))
    inflow = solve_perimeter_graph(tiles, rows, cols, int(tile_rows), int(tile_cols), perim)
    for t in range(len(tiles)):
        fac, _ = engine.accumulate(load(t), inflow[t], False)
        write_window(tiles[t][0], tiles[t][2], fac)
    return len(tiles)


def flow_accumulation_file_tiled(input_path, output_path, tile_rows, tile_cols=None, engine=None, device=None):
    """File-level form: band 1 of a flow-direction GeoTIFF in, a 1-band Int64 GeoTIFF out (the conventions of
    flow_accumulation.flow_accumulation), the host holding one tile at a time."""
    from .constants import FLOW_ACCUMULATION_NODATA
    from .util import raster as _raster

    tile_cols = tile_rows if tile_cols is None else tile_cols
    src = _raster.open_raster(input_path)
    band = src.GetRasterBand(1)
    rows, cols = band.YSize, band.XSize
    dst = _raster.create_raster(output_path, cols, rows, "Int64", projection=src.GetProjection(),
                                geotransform=src.GetGeoTransform())
    out_band = dst.GetRasterBand(1)
    out_band.SetNoDataValue(FLOW_ACCUMULATION_NODATA)
    n = flow_accumulation_tiled(
        lambda r0, r1, c0, c1: band.ReadAsArray(xoff=c0, yoff=r0, win_xsize=c1 - c0, win_ysize=r1 - r0),
        lambda r0, c0, fac: out_band.WriteArray(fac, xoff=c0, yoff=r0),
        rows, cols, tile_rows, tile_cols, engine=engine, device=device)
    dst.FlushCache()
    dst = None
    return n
