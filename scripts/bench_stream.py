#!/usr/bin/env python
"""File-to-file timing of the streaming drivers (SURVEY 8f rank 1) and of out-of-core accumulation (rank 3).

    python scripts/bench_stream.py [--size 32768] [--dir /tmp] [--band-rows N] [--out-of-core]

Generates the synthetic benchmark DEM on the device, writes it as a (Big)TIFF, then times
DEM file -> codes file + counts file through the band pipeline, and codes file -> counts file through the same
pipeline, and prints one JSON line with both stage breakdowns.  Each timed run follows one untimed run that warms
the files.  Both counts files are compared band by band with the device counts of the same DEM (computed before
the timed runs).  The files live under --dir; /dev/shm measures the pipeline without a disk, a real directory
measures it with one.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=32768)
    ap.add_argument("--dir", default="/tmp")
    ap.add_argument("--band-rows", type=int, default=None)
    ap.add_argument("--out-of-core", action="store_true", help="also time flow_accumulation_file_out_of_core")
    ap.add_argument("--strip-rows", type=int, default=4096)
    args = ap.parse_args()
    import numpy as np
    import torch

    from overflow_b200 import device as dev, streaming, strips
    from overflow_b200.util.raster import create_raster, open_raster

    S = args.size
    d = os.path.join(args.dir, f"ofl_stream_{os.getpid()}")
    os.makedirs(d, exist_ok=True)
    p = lambda n: os.path.join(d, n)  # noqa: E731
    out = {"size": S, "dir": args.dir}
    try:
        dem = dev.synth_dem(S, S, seed=0, kind=0, holes_permille=5)
        t0 = time.perf_counter()
        ds = create_raster(p("dem.tif"), S, S, "Float32", geotransform=(0.0, 10.0, 0.0, 0.0, 0.0, -10.0))
        b = ds.GetRasterBand(1)
        for r in range(0, S, 2048):
            b.WriteArray(dem[r : r + 2048].cpu().numpy(), xoff=0, yoff=r)
        b.SetNoDataValue(-9999.0)
        ds.FlushCache()
        ds = b = None
        out["write_dem_s"] = time.perf_counter() - t0
        want_fac = dev.flow_routing(dem, -9999.0)[1].cpu().numpy()  # the exactness reference, off the device
        del dem
        torch.cuda.empty_cache()
        for _ in range(2):  # the first run warms the files
            rep = streaming.stream_routing(p("dem.tif"), p("fdr_s.tif"), p("fac_s.tif"), band_rows=args.band_rows)
        out["streamed"] = rep
        for _ in range(2):
            rep = streaming.stream_accumulation(p("fdr_s.tif"), p("fac_a.tif"), band_rows=args.band_rows)
        out["accumulation"] = rep
        for key, fac_file in (("streamed", "fac_s.tif"), ("accumulation", "fac_a.tif")):
            a = open_raster(p(fac_file)).GetRasterBand(1)
            out[key]["Gcells_per_s"] = S * S / out[key]["wall_s"] / 1e9
            out[key]["equals_device"] = all(
                np.array_equal(a.ReadAsArray(xoff=0, yoff=r, win_xsize=S, win_ysize=min(2048, S - r)),
                               want_fac[r : r + 2048]) for r in range(0, S, 2048))
        del want_fac
        if args.out_of_core:
            t0 = time.perf_counter()
            n = strips.flow_accumulation_file_out_of_core(p("fdr_s.tif"), p("fac_o.tif"), args.strip_rows)
            wall = time.perf_counter() - t0
            a = open_raster(p("fac_s.tif")).GetRasterBand(1)
            c = open_raster(p("fac_o.tif")).GetRasterBand(1)
            same = all(np.array_equal(a.ReadAsArray(xoff=0, yoff=r, win_xsize=S, win_ysize=min(2048, S - r)),
                                      c.ReadAsArray(xoff=0, yoff=r, win_xsize=S, win_ysize=min(2048, S - r)))
                       for r in range(0, S, 2048))
            out["out_of_core"] = {"strips": n, "strip_rows": args.strip_rows, "wall_s": wall,
                                  "Gcells_per_s": S * S / wall / 1e9, "equals_whole_raster": bool(same)}
    finally:
        for f in os.listdir(d):
            os.remove(os.path.join(d, f))
        os.rmdir(d)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
