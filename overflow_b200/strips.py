"""Row-strip (multi-GPU) flow direction + flow accumulation.

The raster is split into contiguous row strips, one per GPU (one process per GPU, torch.distributed).
Per step:
  1. DEM halo exchange   each strip sends its first / last row to the neighbour above / below
                         (NCCL send/recv over NVLink); the raster's top and bottom get nodata rows
  2. direction           strip-mode stencil on the strip + halo rows
  3. code halo exchange  same pattern with the uint8 direction codes
  4. local accumulation  ofl_strip_accum_local: strip-local solve, boundary record block of the strip's
                         first and last row (13 B per boundary cell)
  5. all-gather          the record blocks of all strips (ONE NCCL all_gather, a few MB)
  6. boundary solve      ofl_strip_boundary_solve, replicated on every GPU
  7. final accumulation  ofl_strip_accum_final: push the inflow from other strips down the strip and
                         write the strip's final int64 counts
  8. status              the error flags of 4-7, MAX-reduced over the ranks: the step's one host synchronisation
This mirrors the tile structure of Barnes 2016 (the paper cited by the reference at
src/overflow/flow_accumulation.py:61,100) one level up: strips play the role of tiles.

The compute lives behind a small engine interface so the host-side exchange logic can be tested on
CPU (gloo) with a stand-in engine; the shipped engine (CudaStripEngine) is the C ABI and has no
CPU fallback.
"""
import numpy as np
import torch

from . import _native, device as dev
from .flow_accumulation import as_codes

TILE = 64  # strips must start on multiples of the accumulation tile side


def partition_rows(rows, world, tile=TILE):
    """[(r0, r1)] per rank: contiguous strips whose boundaries are multiples of `tile`.

    Whole tile rows are dealt out as evenly as possible; a ragged remainder (rows % tile) stays with the
    last strip, so every strip has at least `tile` rows.
    """
    n_full = rows // tile
    if n_full < world:
        raise ValueError(f"{rows} rows hold {n_full} full tile rows of {tile}, fewer than {world} strips")
    base, rem = divmod(n_full, world)
    out, t0 = [], 0
    for i in range(world):
        t1 = t0 + base + (1 if i < rem else 0)
        out.append((t0 * tile, rows if i == world - 1 else t1 * tile))
        t0 = t1
    return out


def _round_up(v, a):
    return (v + a - 1) // a * a


def record_bytes(cols):
    """Bytes of one strip's boundary record block (ofl_strip_record_bytes): [2][cols] int64 strip-local counts,
    [2][cols] int32 exit links, [2][cols] uint8 codes, zero padding to a multiple of 256."""
    return _round_up(2 * cols * 13, 256)


def record_views(rec, cols):
    """(floc int64, slink int32, bcode uint8) views, each [..., 2, cols], of a record block [rec_bytes] or of the
    gathered blocks [n_strips, rec_bytes] (uint8 tensors)."""
    lead = tuple(rec.shape[:-1])
    floc = rec[..., : 16 * cols].view(torch.int64).reshape(lead + (2, cols))
    slink = rec[..., 16 * cols : 24 * cols].view(torch.int32).reshape(lead + (2, cols))
    bcode = rec[..., 24 * cols : 26 * cols].reshape(lead + (2, cols))
    return floc, slink, bcode


class CudaStripEngine:
    """The product engine: every method is a liboverflow_b200 call on torch CUDA tensors (device.py).  The strip calls
    only enqueue work on torch's current stream; `flags` hands out their error flags."""

    def __init__(self, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("CudaStripEngine needs a CUDA device (there is no CPU fallback)")

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def strip_workspace(self, rows, cols):
        return dev.strip_workspace(rows, cols, self.device)

    def boundary_workspace(self, n_strips, cols):
        return dev.strip_boundary_workspace(n_strips, cols, self.device)

    def synth_dem(self, out, row0, total_rows, seed, kind, holes_permille, nodata, relief=1000.0):
        dev.synth_dem(*out.shape, row0=row0, total_rows=total_rows, seed=seed, kind=kind, relief=relief,
                      holes_permille=holes_permille, nodata=nodata, out=out)

    def direction(self, dem_halo, nodata, fdr_out):
        dev.flow_direction(dem_halo, nodata, mode="strip", out=fdr_out)

    def accum_local(self, fdr_halo, has_above, has_below, fac, ws, rec):
        dev.strip_accum_local(fdr_halo, has_above, has_below, fac, ws, rec)

    def boundary_solve(self, rec_all, cols, J_all, ws):
        dev.strip_boundary_solve(rec_all, cols, J_all, ws)

    def accum_final(self, fdr_halo, has_above, has_below, J_mine, ws, fac):
        dev.strip_accum_final(fdr_halo, has_above, has_below, J_mine, ws, fac)

    def flags(self, ws, rows, cols, bws, n_strips, out):
        dev.strip_collect_flags(ws, rows, cols, bws, n_strips, out)

    def check(self, fdr_halo, fac, fac_above, fac_below):
        return dev.strip_check_accumulation(fdr_halo, fac, fac_above, fac_below)


def raise_for_flags(flags):
    """flags: the four ints of ofl_strip_collect_flags (already reduced over the ranks)."""
    f = [int(v) for v in flags]
    if f[0] == 3:
        raise _native.OverflowB200Error(-1, "shared-memory window above 64 KB: the tile kernel's 16-bit queue does not apply")
    if any(f):
        where = "tile pass" if f[0] else "strip perimeter graph" if f[1] else "strip-boundary graph"
        raise _native.OverflowB200Error(_native.OFL_ERR_CYCLE, f"flow-direction raster contains a cycle ({where}, flags {f})")


class StripPipeline:
    """One rank's strip: buffers, the per-phase compute, and the distributed step."""

    def __init__(self, rows, cols, rank, world, nodata=-9999.0, engine=None, device=None):
        self.rows, self.cols, self.rank, self.world, self.nodata = rows, cols, rank, world, float(nodata)
        self.r0, self.r1 = partition_rows(rows, world)[rank]
        self.h = self.r1 - self.r0
        self.has_above, self.has_below = rank > 0, rank < world - 1
        if engine is None:
            engine = CudaStripEngine(device if device is not None else torch.device("cuda", torch.cuda.current_device()))
        self.engine = e = engine
        h, c = self.h, cols
        # pitched so every row start satisfies the library's alignment contract
        self.dem_halo = e.empty((h + 2, _round_up(c, 4)), torch.float32)[:, :c]
        self.fdr_halo = e.empty((h + 2, _round_up(c, 16)), torch.uint8)[:, :c]
        self.fac = e.empty((h, c), torch.int64)
        self.ws = e.strip_workspace(h, c)
        self.bws = e.boundary_workspace(world, c)
        self.rec_all = e.empty((world, record_bytes(c)), torch.uint8)  # every strip's boundary record, mine at [rank]
        self.rec = self.rec_all[rank]
        self.J_all = e.empty((world, 2, c), torch.int64)
        self.flags = e.empty((4,), torch.int32)
        self._side = None  # side stream + event of the DEM halo exchange (CUDA only, created on first use)
        self._step_start = None
        self.fac_edge = e.empty((2, c), torch.int64)  # the neighbours' boundary counts (recurrence check only)
        self.fdr_halo.zero_()
        self.rec_all.zero_()
        self.fill_edge_halos()  # the raster's own top / bottom halo rows never change

    # ---- data
    @property
    def dem(self):
        return self.dem_halo[1:-1]

    @property
    def fdr(self):
        return self.fdr_halo[1:-1]

    def load_synthetic(self, seed=0, kind=0, holes_permille=0, relief=1000.0):
        self.engine.synth_dem(self.dem, self.r0, self.rows, seed, kind, holes_permille, self.nodata, relief)

    def load_dem(self, dem_strip):
        self.dem.copy_(torch.as_tensor(dem_strip))

    # ---- phases (compute only)
    def fill_edge_halos(self):
        # util/raster.py:67 pads the raster edge with the band nodata cast to the band dtype
        if not self.has_above:
            self.dem_halo[0].fill_(np.float32(self.nodata).item())
        if not self.has_below:
            self.dem_halo[-1].fill_(np.float32(self.nodata).item())

    def fill_fdr_halo_from_dem(self):
        """The neighbouring strips' code rows, as far as the accumulation of THIS strip needs them, from the DEM halo
        rows already here: which of their cells are NODATA (code 9) and which are not (any other code; 0 is
        written).  The strip's first and last rows are followed as edge rows whatever flows into them, a path that
        steps across the boundary only asks whether the cell it lands on is NODATA (pass A's halo classification),
        and everything else about those rows travels in the boundary records.  `check()` fetches the real rows."""
        nd32 = np.float32(self.nodata)
        representable = float(nd32) == float(self.nodata)  # as in the stencil: other values never match (NaN included)
        for k, there in ((0, self.has_above), (-1, self.has_below)):
            if not there:
                continue
            if representable:
                torch.mul(self.dem_halo[k] == nd32.item(), 9, out=self.fdr_halo[k])
            else:
                self.fdr_halo[k].zero_()

    def direction(self, r0=0, r1=None):
        """Codes of strip rows [r0, r1) (default: all); they read DEM rows r0 - 1 .. r1 of the strip."""
        r1 = self.h if r1 is None else r1
        if r1 > r0:
            self.engine.direction(self.dem_halo[r0 : r1 + 2], self.nodata, self.fdr[r0:r1])

    def accum_local(self):
        self.engine.accum_local(self.fdr_halo, self.has_above, self.has_below, self.fac, self.ws, self.rec)

    def boundary_solve(self):
        self.engine.boundary_solve(self.rec_all, self.cols, self.J_all, self.bws)

    def accum_final(self):
        self.engine.accum_final(self.fdr_halo, self.has_above, self.has_below, self.J_all[self.rank], self.ws, self.fac)

    def collect_flags(self):
        self.engine.flags(self.ws, self.h, self.cols, self.bws, self.world, self.flags)

    # ---- distributed step (one process per strip)
    def _exchange_start(self, first, last, above, below):
        """Start sending `first` / `last` (my first / last row of something) to the strip above / below and receiving
        theirs into `above` / `below`; returns the requests (wait on them before touching `above` / `below`)."""
        import torch.distributed as dist

        ops = []
        if self.has_above:
            ops.append(dist.P2POp(dist.isend, first, self.rank - 1))
            ops.append(dist.P2POp(dist.irecv, above, self.rank - 1))
        if self.has_below:
            ops.append(dist.P2POp(dist.isend, last, self.rank + 1))
            ops.append(dist.P2POp(dist.irecv, below, self.rank + 1))
        return dist.batch_isend_irecv(ops) if ops else []

    def _exchange(self, first, last, above, below):
        for req in self._exchange_start(first, last, above, below):
            req.wait()

    def _exchange_halo(self, buf):
        self._exchange(buf[1], buf[-2], buf[0], buf[-1])

    def step(self, check_status=True):
        """flow direction + flow accumulation of the whole raster; this rank's strip ends up in self.fdr / self.fac.

        Everything is enqueued on the current stream: ONE halo exchange (DEM rows), ONE all-gather of the boundary records
        and, with check_status, one MAX all-reduce of the error flags followed by the step's only host
        synchronisation -- every rank then raises the same error (a cyclic raster) instead of one rank leaving the
        others waiting in a collective."""
        import torch.distributed as dist

        if self.world > 1:
            # the DEM halo rows travel while the stencil works on the rows that do not need them
            d = self.dem_halo
            if d.is_cuda:
                # The stencil is launched FIRST, so the device starts at once; the exchange is set up afterwards on a
                # side stream (NCCL orders itself behind the stream that is current), which waits for everything
                # enqueued before this step -- the last readers of the halo rows -- but not for the stencil.
                main = torch.cuda.current_stream(d.device)
                if self._side is None:
                    self._side = torch.cuda.Stream(d.device)
                    self._step_start = torch.cuda.Event()
                self._step_start.record(main)
                self.direction(1, self.h - 1)
                self._side.wait_event(self._step_start)
                with torch.cuda.stream(self._side):
                    self._exchange(d[1], d[-2], d[0], d[-1])
                main.wait_stream(self._side)
            else:
                reqs = self._exchange_start(d[1], d[-2], d[0], d[-1])
                self.direction(1, self.h - 1)
                for req in reqs:
                    req.wait()
            self.direction(0, 1)
            self.direction(self.h - 1, self.h)
            if d.is_cuda:
                self.fill_fdr_halo_from_dem()  # no second exchange on the critical path
            else:
                self._exchange_halo(self.fdr_halo)
        else:
            self.direction()
        self.accum_local()
        if self.world > 1:
            if dist.get_backend() == "gloo":  # CPU tests
                dist.all_gather(list(self.rec_all.unbind(0)), self.rec.clone())
            else:
                dist.all_gather_into_tensor(self.rec_all, self.rec)
        self.boundary_solve()
        self.accum_final()
        if check_status:
            self.collect_flags()
            if self.world > 1:
                dist.all_reduce(self.flags, op=dist.ReduceOp.MAX)
            raise_for_flags(self.flags.tolist())

    def check(self):
        """Cells of this strip that violate the accumulation recurrence, the boundary rows checked against the
        neighbouring strips' counts (exchanged here).  Summed over the strips, zero proves the partitioned result."""
        above = below = None
        if self.world > 1:
            self._exchange_halo(self.fdr_halo)  # the checker reads the neighbours' real codes (step() only keeps their NODATA mask)
            self._exchange(self.fac[0], self.fac[-1], self.fac_edge[0], self.fac_edge[1])
            above = self.fac_edge[0] if self.has_above else None
            below = self.fac_edge[1] if self.has_below else None
        return self.engine.check(self.fdr_halo, self.fac, above, below)


def step_in_process(pipes):
    """Run all strips of one raster inside ONE process (loop-back exchange): single-GPU emulation of
    the multi-GPU path for tests, and the way to check N-strip == 1-strip results."""
    world = len(pipes)

    def exchange(get):
        for i, p in enumerate(pipes):
            if i > 0:
                get(p)[0].copy_(get(pipes[i - 1])[-2])
            if i < world - 1:
                get(p)[-1].copy_(get(pipes[i + 1])[1])

    for p in pipes:
        p.fill_edge_halos()
    exchange(lambda p: p.dem_halo)
    for p in pipes:
        p.direction()
    if pipes[0].dem_halo.is_cuda:
        for p in pipes:
            p.fill_fdr_halo_from_dem()  # what step() does instead of a second exchange
    else:
        exchange(lambda p: p.fdr_halo)
    for p in pipes:
        p.accum_local()
    for p in pipes:
        for i, q in enumerate(pipes):
            if i != p.rank:
                p.rec_all[i].copy_(q.rec)
    for p in pipes:
        p.boundary_solve()
        p.accum_final()
    for p in pipes:
        p.collect_flags()
        raise_for_flags(p.flags.tolist())


def check_in_process(pipes):
    """Recurrence violations of all strips of step_in_process (loop-back exchange of the boundary counts)."""
    bad = 0
    for i, p in enumerate(pipes):  # the checker reads the neighbours' real code rows
        if i > 0:
            p.fdr_halo[0].copy_(pipes[i - 1].fdr_halo[-2])
        if i < len(pipes) - 1:
            p.fdr_halo[-1].copy_(pipes[i + 1].fdr_halo[1])
    for i, p in enumerate(pipes):
        above = pipes[i - 1].fac[-1].contiguous() if i > 0 else None
        below = pipes[i + 1].fac[0].contiguous() if i < len(pipes) - 1 else None
        bad += p.engine.check(p.fdr_halo, p.fac, above, below)
    return bad


# ---------------------------------------------------------------- out of core: strips through ONE device
def strip_bounds(rows, strip_rows, tile=TILE):
    """[(r0, r1)]: consecutive strips of `strip_rows` rows (a multiple of the tile side).  A remainder of less than
    one tile row stays with the last strip (as in partition_rows: the library wants at least two rows per strip)."""
    strip_rows = int(strip_rows)
    if strip_rows < tile or strip_rows % tile:
        raise ValueError(f"strip_rows must be a positive multiple of {tile}, got {strip_rows}")
    out = [(r0, min(rows, r0 + strip_rows)) for r0 in range(0, rows, strip_rows)]
    if len(out) > 1 and out[-1][1] - out[-1][0] < tile:
        out[-2:] = [(out[-2][0], rows)]
    return out


def flow_accumulation_out_of_core(read_rows, write_rows, rows, cols, strip_rows, engine=None, device=None):
    """Flow accumulation of a flow-direction raster that need not fit the device (SURVEY 8f rank 3, full-width
    tiles): the raster goes through ONE device strip by strip, twice, in the structure of Barnes 2016 that the
    multi-GPU path uses across devices.

        read_rows(r0, r1)  -> uint8 array [r1 - r0, cols] with the codes of those rows (any host source: an array,
                              a memmap, a raster band)
        write_rows(r0, fac)   receives the final int64 counts of rows r0 .. r0 + len(fac) (a host array it may keep)

    Pass 1 solves every strip on its own and keeps only its boundary records (13 B per boundary cell); the boundary
    graph of all strips is solved on the device; pass 2 solves each strip again (nothing of pass 1 is kept but the
    records) and pushes the inflow from the other strips down before the counts leave.  Device memory: one strip
    (codes, counts, workspace) plus 26 B x cols x strips of records.  The result equals the whole-raster
    accumulation bit for bit (integer sums).  Returns the number of strips.
    """
    if engine is None:
        engine = CudaStripEngine(device if device is not None else torch.device("cuda", torch.cuda.current_device()))
    e = engine
    bounds = strip_bounds(rows, strip_rows)
    n = len(bounds)
    h_max = max(r1 - r0 for r0, r1 in bounds)
    fdr_halo = e.empty((h_max + 2, _round_up(cols, 16)), torch.uint8)[:, :cols]
    fac = e.empty((h_max, cols), torch.int64)
    ws = e.strip_workspace(h_max, cols)
    rec_all, J_all = e.empty((n, record_bytes(cols)), torch.uint8), e.empty((n, 2, cols), torch.int64)
    scratch = e.empty((record_bytes(cols),), torch.uint8)
    bws = e.boundary_workspace(n, cols)
    flags = e.empty((4,), torch.int32)

    def status(ws_, rows_, bws_):
        e.flags(ws_, rows_, cols, bws_, n, flags)
        raise_for_flags(flags.tolist())

    def load(s):
        """Codes of strip s plus one halo row above and below (raster edges: the halo row is never looked at)."""
        r0, r1 = bounds[s]
        lo, hi = max(0, r0 - 1), min(rows, r1 + 1)
        block = as_codes(read_rows(lo, hi))
        if block.shape != (hi - lo, cols):
            raise ValueError(f"read_rows({lo}, {hi}) returned shape {block.shape}, expected {(hi - lo, cols)}")
        view = fdr_halo[: r1 - r0 + 2]
        view[(lo - r0 + 1) : (hi - r0 + 1)].copy_(torch.from_numpy(block))
        if lo == r0:
            view[0].zero_()
        if hi == r1:
            view[-1].zero_()
        return view, fac[: r1 - r0], s > 0, s < n - 1

    for s in range(n):
        view, f, above, below = load(s)
        e.accum_local(view, above, below, f, ws, rec_all[s])
        status(ws, f.shape[0], None)
    e.boundary_solve(rec_all, cols, J_all, bws)
    status(None, 0, bws)
    for s in range(n):
        view, f, above, below = load(s)
        e.accum_local(view, above, below, f, ws, scratch)
        e.accum_final(view, above, below, J_all[s], ws, f)
        status(ws, f.shape[0], None)
        write_rows(bounds[s][0], f.cpu().numpy())
    return n


def flow_accumulation_file_out_of_core(input_path, output_path, strip_rows, engine=None, device=None):
    """File-level form of flow_accumulation_out_of_core: band 1 of a flow-direction GeoTIFF in, a 1-band Int64
    GeoTIFF out (same conventions as flow_accumulation.flow_accumulation), with the host holding one strip at a time."""
    from .constants import FLOW_ACCUMULATION_NODATA
    from .util import raster as _raster

    src = _raster.open_raster(input_path)
    band = src.GetRasterBand(1)
    rows, cols = band.YSize, band.XSize
    dst = _raster.create_raster(output_path, cols, rows, "Int64", projection=src.GetProjection(),
                                geotransform=src.GetGeoTransform())
    out_band = dst.GetRasterBand(1)
    out_band.SetNoDataValue(FLOW_ACCUMULATION_NODATA)
    n = flow_accumulation_out_of_core(
        lambda r0, r1: band.ReadAsArray(xoff=0, yoff=r0, win_xsize=cols, win_ysize=r1 - r0),
        lambda r0, fac: out_band.WriteArray(fac, xoff=0, yoff=r0),
        rows, cols, strip_rows, engine=engine, device=device)
    dst.FlushCache()
    dst = None
    return n
