"""Streaming file drivers: GeoTIFF -> device -> GeoTIFF with file reads, PCIe copies, kernels and file writes
overlapped (SURVEY 8f rank 1).

The reference's `flow_direction()` (src/overflow/flow_direction.py:99-124) reads a chunk, computes it, writes it,
one after the other (util/raster.py:174-210).  Here the raster moves in ROW BANDS through a pipeline

    reader thread -> pinned ring -> H2D (copy stream) -> kernels (compute stream) -> D2H (copy stream)
                  -> pinned ring -> writer thread

so that the wall-clock time tends to max(file I/O, PCIe) instead of their sum.  Semantics are the reference's:
band 1 of the input, the band's nodata value required (util/raster.py:59), out-of-raster neighbours read as
nodata (util/raster.py:67), outputs are 1-band GeoTIFFs with the input's projection and geotransform -- Byte with
nodata 9 for the codes, Int64 with nodata FLOW_ACCUMULATION_NODATA for the counts.

One pipeline serves both inputs.  A DEM goes up into a device DEM with a nodata halo row above and below, and the
direction stencil runs per band as soon as the band below it has arrived; flow-direction codes go up straight into
the device codes.  The whole raster is resident on the device between the two kernels (accumulation needs every
code before it can finish a single count); rasters beyond device memory take
`strips.flow_accumulation_file_out_of_core`.  The accumulation runs once, after the last band (at 64k x 64k it is
25 ms next to tens of seconds of I/O -- splitting it per band would buy nothing).
PyTorch owns device memory, pinned memory and streams here; every kernel is in liboverflow_b200.
"""
import queue
import threading
import time

import numpy as np

from . import _native
from .constants import FLOW_ACCUMULATION_NODATA, FLOW_DIRECTION_NODATA
from .flow_accumulation import as_codes


def _get(q, check):
    """`q.get()` that calls `check` every 0.1 s while it waits; `check` raises once the item can no longer come."""
    while True:
        try:
            return q.get(timeout=0.1)
        except queue.Empty:
            check()


class _Worker(threading.Thread):
    """A thread that runs jobs from a queue in order.  After a job raises, or once `stop` is set, the remaining
    jobs are dropped; the exception is kept in `error` for the caller to raise."""

    def __init__(self, name, stop):
        super().__init__(name=name, daemon=True)
        self.jobs = queue.Queue()
        self.stop = stop
        self.error = None
        self.busy_s = 0.0  # time spent in the file I/O calls themselves (the jobs report it; waits are not counted)
        self.start()

    def run(self):
        for job in iter(self.jobs.get, None):
            if self.error is None and not self.stop.is_set():
                try:
                    job()
                except BaseException as e:  # noqa: BLE001 -- handed to the main thread
                    self.error = e

    def submit(self, job):
        self.jobs.put(job)

    def close(self):
        """End the thread once the jobs queued so far have run (or have been dropped)."""
        self.jobs.put(None)
        self.join()


def _read_rows_into(band, r0, r1, out):
    """Rows [r0, r1) of the band into the (pinned) array `out`, without a second host copy where the band can."""
    try:
        res = band.ReadAsArray(xoff=0, yoff=r0, win_xsize=band.XSize, win_ysize=r1 - r0, buf_obj=out)
        if res is not out:
            out[...] = res
    except TypeError:  # a band without buf_obj
        out[...] = band.ReadAsArray(xoff=0, yoff=r0, win_xsize=band.XSize, win_ysize=r1 - r0)


def _write_job(writer, event, out_band, ring, slot, r0, r1):
    """Writer-thread job: wait for the band's D2H copy, write rows [r0, r1), hand the pinned buffer back."""
    def job():
        event.synchronize()
        t0 = time.perf_counter()
        out_band.WriteArray(ring.bufs[slot].numpy()[: r1 - r0], xoff=0, yoff=r0)
        writer.busy_s += time.perf_counter() - t0
        ring.release(slot)
    return job


class _Ring:
    """`n` pinned host buffers handed round in order; a buffer is reused only after `release` (an event or a
    thread finishing with it)."""

    def __init__(self, torch, n, shape, dtype):
        self.bufs = [torch.empty(shape, dtype=dtype, pin_memory=True) for _ in range(n)]
        self.free = queue.Queue()
        for i in range(n):
            self.free.put(i)

    def acquire(self, check):
        """The next free buffer; `check` is called while none is free (see `_get`)."""
        i = _get(self.free, check)
        return i, self.bufs[i]

    def release(self, i):
        self.free.put(i)


def stream_routing(input_path, flow_direction_path=None, flow_accumulation_path=None, band_rows=None, device=None,
                   ring=3):
    """DEM GeoTIFF -> flow-direction GeoTIFF and / or flow-accumulation GeoTIFF through the band pipeline.

    Either output path may be None (direction only: no accumulation is run; accumulation only: the codes are not
    written).  Returns a dict with the wall-clock time and the busy time of every pipeline stage.
    The DEM band must be Float32 (other dtypes take flow_routing()'s read-all path, whose generic stencil they need).
    """
    if flow_direction_path is None and flow_accumulation_path is None:
        raise ValueError("nothing to write: give a flow-direction and / or a flow-accumulation path")
    return _stream(input_path, True, flow_direction_path, flow_accumulation_path, band_rows, device, ring)


def stream_accumulation(input_path, output_path, band_rows=None, device=None, ring=3):
    """Flow-direction GeoTIFF -> flow-accumulation GeoTIFF: the codes go up in bands while the file is still being
    read, the counts come down in bands while the file is being written (same output as flow_accumulation()).
    Returns the same report as `stream_routing`."""
    return _stream(input_path, False, None, output_path, band_rows, device, ring)


def _stream(input_path, dem_in, flow_direction_path, flow_accumulation_path, band_rows, device, ring):
    """The band pipeline; `dem_in`: the input is a DEM (else flow-direction codes)."""
    import torch

    from . import device as dev
    from .util import raster as _raster

    t_wall = time.perf_counter()
    src = _raster.open_raster(input_path)
    band = src.GetRasterBand(1)
    rows, cols = band.YSize, band.XSize
    in_dtype = _raster.gdal_data_type_to_numpy_data_type(band.DataType)
    if dem_in:
        nodata = band.GetNoDataValue()
        assert nodata is not None, "The raster band has no no data value"  # util/raster.py:59 in the reference
        if in_dtype != np.float32:
            raise TypeError("the streaming driver takes Float32 DEMs; other band types go through flow_routing()")
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if device.type != "cuda":
        raise ValueError("the streaming driver needs a CUDA device (there is no CPU fallback)")
    _native.init(device.index if device.index is not None else torch.cuda.current_device())
    up_dtype = torch.float32 if dem_in else torch.uint8  # what a cell is in the input ring and on the device
    cell = up_dtype.itemsize
    if band_rows is None:
        band_rows = max(64, min(16384 // cell, (256 << 20) // max(1, cols * cell)))  # about 256 MiB of input per band
    band_rows = max(1, min(int(band_rows), max(rows, 1)))  # the pinned rings are sized by it
    bands = [(r, min(rows, r + band_rows)) for r in range(0, rows, band_rows)]
    fac_rows = max(1, band_rows * cell // 8)  # 8 B/cell: the counts ring holds as many pinned bytes as the input ring

    def make_out(path, name, nd):
        if path is None:
            return None, None
        ds = _raster.create_raster(path, cols, rows, name, projection=src.GetProjection(), geotransform=src.GetGeoTransform())
        b = ds.GetRasterBand(1)
        b.SetNoDataValue(nd)
        return ds, b

    stop = threading.Event()
    workers = []
    try:
        fdr_ds, fdr_band = make_out(flow_direction_path, "Byte", FLOW_DIRECTION_NODATA)
        fac_ds, fac_band = make_out(flow_accumulation_path, "Int64", FLOW_ACCUMULATION_NODATA)
        with torch.cuda.device(device):
            s_comp = torch.cuda.current_stream(device)
            s_up, s_down = torch.cuda.Stream(device), torch.cuda.Stream(device)
            if dem_in:
                # the DEM carries one nodata row above and below (what util/raster.py:67 pads)
                dem_halo = dev.pitched(rows + 2, cols, torch.float32, device)
                dem_halo[0].fill_(float(np.float32(nodata)))
                dem_halo[-1].fill_(float(np.float32(nodata)))
            fdr = dev.pitched(rows, cols, torch.uint8, device)
            s_up.wait_stream(s_comp)  # the new blocks may still be in use by work queued on s_comp
            in_ring = _Ring(torch, ring, (band_rows, cols), up_dtype)
            code_ring = _Ring(torch, ring, (band_rows + 1, cols), torch.uint8) if fdr_band is not None else None
            workers += [_Worker(name, stop) for name in ("ofl-reader", "ofl-recycle", "ofl-writer")]
            reader, recycler, writer = workers
            filled = queue.Queue()
            ev_t = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
            up_events, dir_events, down_events = [], [], []
            setup_s = time.perf_counter() - t_wall  # files opened / created, device rasters and pinned rings allocated

            def check():  # main thread: raise the first worker error
                for w in workers:
                    if w.error is not None:
                        raise w.error

            def stopped():  # worker threads: give up a wait once the pipeline is being torn down
                if stop.is_set():
                    raise RuntimeError("band pipeline stopped")

            def read_job(b):
                def job():
                    i, buf = in_ring.acquire(stopped)
                    r0, r1 = bands[b]
                    view = buf.numpy()[: r1 - r0]
                    t0 = time.perf_counter()
                    if in_dtype == view.dtype:
                        _read_rows_into(band, r0, r1, view)
                    else:  # codes stored in a wider integer type (the reference's tests use int64 arrays)
                        view[...] = as_codes(band.ReadAsArray(xoff=0, yoff=r0, win_xsize=cols, win_ysize=r1 - r0))
                    reader.busy_s += time.perf_counter() - t0
                    filled.put((b, i))
                return job

            for b in range(len(bands)):
                reader.submit(read_job(b))

            done = 0  # output rows whose codes exist
            for _ in range(len(bands)):
                b, slot = _get(filled, check)
                r0, r1 = bands[b]
                e0, e1 = ev_t(), ev_t()
                with torch.cuda.stream(s_up):
                    e0.record()
                    (dem_halo[1 + r0 : 1 + r1] if dem_in else fdr[r0:r1]).copy_(
                        in_ring.bufs[slot][: r1 - r0], non_blocking=True)
                    e1.record()
                up_events.append((e0, e1))
                recycler.submit((lambda ev, i: (lambda: (ev.synchronize(), in_ring.release(i))))(e1, slot))
                if not dem_in:
                    continue
                # codes of the rows whose three input rows are on the device now
                end = rows if r1 == rows else r1 - 1
                if end > done:
                    s_comp.wait_event(e1)
                    d0, d1 = ev_t(), ev_t()
                    d0.record(s_comp)
                    with torch.cuda.stream(s_comp):  # the slices are pitched already: no copy
                        dev.flow_direction(dem_halo[done : end + 2], nodata, mode="strip", out=fdr[done:end])
                    d1.record(s_comp)
                    dir_events.append((d0, d1))
                    if fdr_band is not None:
                        ci, cbuf = code_ring.acquire(check)
                        c0, c1 = ev_t(), ev_t()
                        with torch.cuda.stream(s_down):
                            s_down.wait_event(d1)
                            c0.record()
                            cbuf[: end - done].copy_(fdr[done:end], non_blocking=True)
                            c1.record()
                        down_events.append((c0, c1))
                        writer.submit(_write_job(writer, c1, fdr_band, code_ring, ci, done, end))
                    done = end
            s_comp.wait_stream(s_up)
            # Every stencil launch waits on s_comp for its band's upload, so the DEM's block can go back to s_comp's
            # pool before the counts and the accumulation workspace are allocated.
            dem_halo = None
            acc_events = None
            if fac_band is not None:
                fac = torch.empty((rows, cols), dtype=torch.int64, device=device)
                a0, a1 = ev_t(), ev_t()
                a0.record(s_comp)
                dev.flow_accumulation(fdr, out=fac)  # pass A, perimeter-graph solve, final pass; raises on a cyclic raster
                a1.record(s_comp)
                acc_events = (a0, a1)
                fac_ring = _Ring(torch, ring, (fac_rows, cols), torch.int64)
                for a in range(0, rows, fac_rows):
                    e = min(rows, a + fac_rows)
                    fi, fbuf = fac_ring.acquire(check)
                    c0, c1 = ev_t(), ev_t()
                    with torch.cuda.stream(s_down):
                        s_down.wait_event(a1)
                        c0.record()
                        fbuf[: e - a].copy_(fac[a:e], non_blocking=True)
                        c1.record()
                    down_events.append((c0, c1))
                    writer.submit(_write_job(writer, c1, fac_band, fac_ring, fi, a, e))
            for w in workers:
                w.close()
            check()
            torch.cuda.synchronize(device)
            t_flush = time.perf_counter()
            for ds in (fdr_ds, fac_ds):
                if ds is not None:
                    ds.FlushCache()  # the written pages reach the file system here (memory-mapped outputs)
            flush_s = time.perf_counter() - t_flush
            wall = time.perf_counter() - t_wall
    finally:
        stop.set()
        for w in workers:
            w.close()
        torch.cuda.synchronize(device)  # no copy may still target a pinned ring when it is dropped below
        # An exception's traceback keeps this frame alive: let go of the files, rings and device rasters now.
        src = band = fdr_ds = fdr_band = fac_ds = fac_band = None
        in_ring = code_ring = fac_ring = dem_halo = fdr = fac = None
    ms = lambda evs: sum(a.elapsed_time(b) for a, b in evs)  # noqa: E731
    cells = rows * cols
    h2d_bytes = cells * cell
    d2h_bytes = (cells if flow_direction_path is not None else 0) + (cells * 8 if flow_accumulation_path is not None else 0)
    report = {
        "rows": rows, "cols": cols, "bands": len(bands), "band_rows": band_rows, "wall_s": wall,
        "setup_s": setup_s, "flush_s": flush_s, "pipeline_s": wall - setup_s - flush_s,
        "read_busy_s": reader.busy_s, "write_busy_s": writer.busy_s,
        "h2d_s": ms(up_events) / 1e3, "d2h_s": ms(down_events) / 1e3,
        "direction_kernel_s": ms(dir_events) / 1e3,
        "accumulation_s": (acc_events[0].elapsed_time(acc_events[1]) / 1e3) if acc_events else 0.0,
        "h2d_bytes": h2d_bytes, "d2h_bytes": d2h_bytes,
        "file_bytes_read": cells * np.dtype(in_dtype).itemsize, "file_bytes_written": d2h_bytes,
    }
    stages = {k: report[k] for k in ("read_busy_s", "write_busy_s", "h2d_s", "d2h_s")}
    report["slowest_stage"] = max(stages, key=stages.get)
    report["pipeline_over_slowest_stage"] = report["pipeline_s"] / max(1e-9, max(stages.values()))
    report["serial_sum_s"] = sum(stages.values()) + report["direction_kernel_s"] + report["accumulation_s"]
    return report
