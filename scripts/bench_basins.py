"""Time drainage-basin labelling (ofl_label_basins_u8, device buffers) on synthetic DEMs, next to the accumulation of
the same codes.

    python scripts/bench_basins.py --out basins.json [--size 65536] [--kind 0 1 2 3 4] [--calls 10] [--warmup 2]

Per kind: the DEM is generated on the device and its codes computed there; then, in one process, ms per labelling call
(CUDA events, median over --calls calls after --warmup), the per-phase split (a separate run with phase timing on),
Gcells/s, algorithmic GB/s at 9 B/cell (1 B codes in, 8 B labels out) and its share of the HBM peak, the checker's
violation count (must be 0) and the accumulation's ms per call on the same codes.  At sizes up to 16384^2 the label
count of every outlet is also compared with the accumulation's count there.  The card's name and power limit are
recorded with the numbers.  Writes one JSON document to --out and prints it.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from overflow_b200 import _native, device as dev  # noqa: E402

BYTES_PER_CELL = 9.0
NODATA = -9999.0


def card():
    res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True)
    name, power = res.stdout.strip().splitlines()[0].split(", ")
    return {"name": name, "power_limit": power}


def timed(fn, calls, warmup):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(calls):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), times


def outlet_sizes_match(fdr, labels, fac):
    flat = labels.reshape(-1)
    idx = torch.arange(flat.numel(), device=flat.device, dtype=torch.int64)
    outlet = flat == idx + 1
    counts = torch.bincount(flat, minlength=flat.numel() + 1)
    return bool(torch.equal(counts[idx[outlet] + 1], fac.reshape(-1)[outlet]))


def run_kind(n, kind, calls, warmup, peak):
    dem = dev.synth_dem(n, n, seed=3, kind=kind, holes_permille=5 if kind in (0, 1) else 0)
    fdr = dev.flow_direction(dem, NODATA)
    del dem
    torch.cuda.empty_cache()
    labels = torch.empty((n, n), dtype=torch.int64, device="cuda")
    ws = dev.basins_workspace(n, n)
    ms, times = timed(lambda: dev.label_basins(fdr, out=labels, workspace=ws), calls, warmup)
    _native.phase_timing_read(reset=True)
    _native.phase_timing_enable(True)
    for _ in range(3):
        dev.label_basins(fdr, out=labels, workspace=ws)
    torch.cuda.synchronize()
    ph = _native.phase_timing_read(reset=True)
    _native.phase_timing_enable(False)
    phases = {k: ph[k][0] / 3 for k in ("basins_tile", "basins_solve", "basins_final")}
    bad = dev.check_basins(fdr, labels)
    outlets = int((labels.reshape(-1) == torch.arange(1, n * n + 1, device="cuda", dtype=torch.int64)).sum())
    del ws
    if n <= 16384:
        fac = torch.empty((n, n), dtype=torch.int64, device="cuda")
    else:  # 65536^2: the counts go into the labels' buffer once the labels are checked
        fac = labels
    acc_ws = dev.accumulation_workspace(n, n)
    acc_ms, _ = timed(lambda: dev.flow_accumulation(fdr, out=fac, workspace=acc_ws), calls, warmup)
    sizes = outlet_sizes_match(fdr, labels, fac) if fac is not labels else None
    cells = n * n
    gbs = cells * BYTES_PER_CELL / ms / 1e6
    return {
        "size": n, "kind": kind, "ms": ms, "ms_all": times, "phases_ms": phases, "gcells_s": cells / ms / 1e6,
        "algorithmic_gbs_9B": gbs, "frac_of_hbm_peak": gbs / peak, "check_violations": bad, "outlets": outlets,
        "outlet_sizes_equal_fac": sizes, "accumulation_ms": acc_ms,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON output path")
    ap.add_argument("--size", type=int, default=65536)
    ap.add_argument("--kind", type=int, nargs="+", default=[0, 1, 2, 3, 4])
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_basins.py needs a CUDA device")
    peak = 6551.4
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    _native.init(0)
    doc = {"what": "ofl_label_basins_u8, device buffers; accumulation_ms: ofl_flow_accumulation_u8 on the same codes",
           "card": card(), "hbm_peak_gbs": peak, "runs": []}
    for kind in a.kind:
        doc["runs"].append(run_kind(a.size, kind, a.calls, a.warmup, peak))
        torch.cuda.empty_cache()
        print(json.dumps(doc["runs"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
