#!/usr/bin/env python
"""bench.py -- D8 flow direction + flow accumulation throughput on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--size S] [--dump-outputs DIR]

One step = one pass of the hot path (flow direction, then flow accumulation) over one synthetic
float32 DEM.  N=1: the S x S raster (default 65536, BASELINE.json configs[2]) is resident in HBM
and processed by one GPU.  N>1 (launched by torchrun, one rank per GPU): the same raster split into
N row strips (strong scaling), halo rows and the strip-boundary records exchanged over NCCL.
`--impl reference` times the reference's algorithm on the host cores (the CPU port in oracle/, plus the
reference's own numba direction kernel when oracle/_ref holds it) on a bounded sample of the same DEM.
Prints ONE JSON line on rank 0.

Every number that leaves this file is checked on the benchmarked result itself (`parity`): the accumulation
recurrence on every cell (across strip boundaries too), 64-bit position-weighted checksums of every strip
against the same rows of a single-GPU run of the whole raster (N>1), and oracle-checked direction windows
that touch the strip boundaries.  `other_workloads` repeats step + checks on the flat-heavy and the
adversarial long-path DEMs (BASELINE.json configs[3], configs[4]).

`--dump-outputs DIR` writes what the timed path returned in its last timed step -- codes and counts at a fixed,
seeded sample of cells (every cell of a small raster) -- so that two builds, or two GPU counts, can be compared output
for output on identical inputs.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NODATA = -9999.0
METRIC = "d8_flowdir_flowacc_throughput"
UNIT = "Gcells/s"
DIR_BYTES_PER_CELL = 5.0   # 4 B float32 read + 1 B code write            (SURVEY 8d)
ACC_BYTES_PER_CELL = 9.0   # 1 B code read + 8 B int64 count write         (SURVEY 8d)
HBM_NOMINAL_GBS = 8000.0   # nominal HBM3e bandwidth of a B200 (SURVEY 8d: report against the measured peak and this one)
# accumulation: 9 B/cell = 1 B code read (pass A) + 8 B count write (final pass)
PHASE_BYTES = {"direction": 5.0, "acc_tile_a": 1.0, "acc_tile_b": 8.0}
KINDS = {0: "fractal value-noise", 1: "terraced fractal", 2: "tilted plane", 3: "walled serpentine (one channel, east-west runs)",
         4: "walled serpentine (one channel, north-south runs)"}
# --dump-outputs: cells written per raster, 40 MB in all (codes float32, counts and cell indices float64), under 64 MB
DUMP_CELLS = 1 << 21
DUMP_SEED = 0


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------- --dump-outputs
def dump_cells(rows, cols):
    """Row-major indices of the cells --dump-outputs writes, ascending: every cell of a raster of at most DUMP_CELLS
    cells, else DUMP_CELLS distinct cells drawn with a fixed seed (the same for every run, build and GPU count)."""
    import numpy as np

    n = rows * cols
    if n <= DUMP_CELLS:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_CELLS, replace=False))


def dump_outputs(out_dir, fdr, fac, row0, rows, cols, sum_ranks=None):
    """Writes DIR/fdr.npy (codes, float32), DIR/fac.npy (counts, float64) and DIR/cells.npy (their row-major indices,
    float64) for the cells dump_cells(rows, cols) names.  `fdr` / `fac` (numpy arrays or device tensors) hold rows
    row0 .. row0 + len(fdr) of the raster; with several ranks each contributes zeros outside its rows, `sum_ranks`
    adds the ranks' arrays and only the caller passing out_dir writes.  Both conversions are exact."""
    import numpy as np

    cells = dump_cells(rows, cols)
    lo = row0 * cols
    mine = (cells >= lo) & (cells < lo + fdr.shape[0] * cols)
    r, c = np.divmod(cells[mine] - lo, cols)
    if not isinstance(fdr, np.ndarray):  # gather on the device; only the sample is copied to the host
        import torch

        r, c = torch.from_numpy(r).to(fdr.device), torch.from_numpy(c).to(fdr.device)
    out = {"fdr": np.zeros(len(cells), np.float32), "fac": np.zeros(len(cells), np.float64)}
    for name, full in (("fdr", fdr), ("fac", fac)):
        got = full[r, c]
        out[name][mine] = got if isinstance(got, np.ndarray) else got.cpu().numpy()
        if sum_ranks is not None:
            out[name] = sum_ranks(out[name])
    if out_dir is None:
        return
    os.makedirs(out_dir, exist_ok=True)
    out["cells"] = cells.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---------------------------------------------------------------- reference arm (CPU, no CUDA library in the process)
def cpu_pass(oracle, dem_pad, numba_direction=None):
    """Reference algorithm on the host: direction on all threads (prange), accumulation serial."""
    t0 = time.perf_counter()
    if numba_direction is not None:
        fdr = numba_direction(dem_pad, NODATA)[1:-1, 1:-1]
    else:
        fdr = oracle.flow_direction_for_tile(dem_pad, NODATA)[1:-1, 1:-1]
    t1 = time.perf_counter()
    fac = oracle.flow_accumulation(fdr)
    t2 = time.perf_counter()
    return fdr, fac, t1 - t0, t2 - t1


def host_dem_padded(oracle, args, sample):
    """`sample` x `sample` top-left window of the benchmark DEM plus a nodata ring, generated on the HOST by the
    restatement of the device generator (oracle/synth_host.c, bit-identical): the reference arm never maps the
    CUDA library."""
    import numpy as np

    out = np.full((sample + 2, sample + 2), NODATA, dtype=np.float32)
    out[1:-1, 1:-1] = oracle.synth_dem(sample, sample, total_rows=args.size, total_cols=args.size, seed=args.seed,
                                       kind=args.kind, holes_permille=args.holes, nodata=NODATA)
    return out


def reference_numba_direction():
    """The reference's own flow_direction_for_tile (numba, prange over all host threads) when oracle/_ref holds a copy
    of the reference's three Python files (oracle/make_ref.py, run in the dev container); else None."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref, "overflow", "flow_direction.py")):
        return None
    try:
        sys.path.insert(0, ref)
        import importlib

        mod = importlib.import_module("overflow.flow_direction")
        return getattr(mod, "flow_direction_for_tile")
    except Exception:
        return None
    finally:
        if ref in sys.path:
            sys.path.remove(ref)


def repo_libraries_loaded():
    """Shared objects under the repository mapped into this process (the reference arm must not map the CUDA library)."""
    try:
        with open("/proc/self/maps") as f:
            return sorted({ln.split()[-1] for ln in f if ".so" in ln and ROOT in ln})
    except OSError:
        return []


def run_reference(args):
    """--impl reference: the reference's path on the box's host cores, on a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle

    oracle.build()
    # every host thread this process may use, whatever OMP_NUM_THREADS says (torchrun sets it to 1 for N > 1)
    try:
        n_thr = len(os.sched_getaffinity(0))
    except AttributeError:
        n_thr = os.cpu_count() or 1
    oracle.set_num_threads(n_thr)
    sample = min(args.size, args.cpu_sample)
    dem_pad = host_dem_padded(oracle, args, sample)
    numba_dir = None
    if not args.no_numba:
        os.environ.setdefault("NUMBA_NUM_THREADS", str(n_thr))
        numba_dir = reference_numba_direction()
    cells = sample * sample
    if numba_dir is not None:
        import numpy as np

        numba_dir(np.ascontiguousarray(dem_pad[:66, :66]), NODATA)  # JIT compile outside the timed region
    for _ in range(args.warmup):
        cpu_pass(oracle, dem_pad, numba_dir)
    t0 = time.perf_counter()
    td = ta = 0.0
    for _ in range(args.steps):
        fdr, fac, a, b = cpu_pass(oracle, dem_pad, numba_dir)
        td += a
        ta += b
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, fdr, fac, 0, sample, sample)
    value = cells * args.steps / el / 1e9
    dir_how = ("the reference's own numba flow_direction_for_tile (oracle/_ref)" if numba_dir is not None
               else "C port (oracle/d8_oracle.c, OpenMP)")
    sample_txt = (f"{sample}x{sample} top-left window of the {args.size}x{args.size} DEM (host generator); direction: "
                  f"{dir_how} on {n_thr} threads {td / args.steps * 1e3:.0f} ms; accumulation: C port with an O(1) FIFO "
                  f"(the reference's list.pop(0) sweep is O(N^2)), serial as in the reference, "
                  f"{ta / args.steps * 1e3:.0f} ms per step")
    cfg = workload_config(args, args.gpus)
    cfg["sample_rows"] = cfg["sample_cols"] = sample
    cfg["sample_note"] = ("the reference arm runs a bounded sample of the workload: rows/cols name the workload, "
                          "sample_rows/sample_cols what was timed; throughput is per cell, so the two arms compare")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32->u8->int64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_thr, "kind": "port",
                         "direction_kind": "reference" if numba_dir is not None else "port", "accumulation_kind": "port",
                         "direction_ms": td / args.steps * 1e3, "accumulation_ms": ta / args.steps * 1e3, "sample": sample_txt},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "repo_libraries_loaded": repo_libraries_loaded(),
    }
    print(json.dumps(line), flush=True)


def workload_config(args, n):
    return {
        "workload": f"flow_direction + flow_accumulation on synthetic {args.size}x{args.size} float32 DEM "
                    f"({KINDS[args.kind]}, {args.holes} permille nodata holes, seed {args.seed})",
        "rows": args.size, "cols": args.size, "partition": f"{n} row strip(s)",
        "cache": "inputs (4 B/cell DEM) far exceed the 126 MB L2, no flush needed",
    }


# ---------------------------------------------------------------- native arm
_K64 = -7046029254386353131  # 0x9E3779B97F4A7C15 as a signed 64-bit value


def checksum(torch, t, row0, total_cols, chunk_rows=1024):
    """64-bit position-weighted checksum of rows row0.. of a raster: sum((v + 1) * ((global index * K) | 1)) mod 2^64.
    Two rasters agree on it only if they agree cell for cell (up to 2^-64); a swap of two cells changes it."""
    rows, cols = t.shape
    total = torch.zeros((), dtype=torch.int64, device=t.device)
    for r in range(0, rows, chunk_rows):
        n = min(chunk_rows, rows - r)
        idx = torch.arange((row0 + r) * total_cols, (row0 + r + n) * total_cols, dtype=torch.int64, device=t.device)
        idx = idx.view(n, total_cols)[:, :cols]
        total += ((t[r : r + n].to(torch.int64) + 1) * ((idx * _K64) | 1)).sum()
    return int(total.item())


def bind_to_gpu_numa(local):
    """Pin this process (and hence its pinned host buffers, first touch) to the NUMA node of its GPU.  Host plumbing
    for the end-to-end leg; returns a short description, or None when the box gives no such information."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bdf = pynvml.nvmlDeviceGetPciInfo(h).busId
        bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return f"numa node {node} ({len(allowed)} cpus)"
    except Exception:
        return None


class SingleRunner:
    """The whole raster on one GPU: one ofl_flow_routing_f32 call per step."""

    def __init__(self, torch, dev, size):
        self.torch, self.dev, self.S = torch, dev, size
        self.dem = dev.synth_dem(size, size, seed=0, kind=2)  # allocates; load() fills
        self.fdr = torch.empty((size, size), dtype=torch.uint8, device="cuda")
        self.fac = torch.empty((size, size), dtype=torch.int64, device="cuda")

    def load(self, seed, kind, holes, relief=1000.0):
        S = self.S
        self.dev.synth_dem(S, S, seed=seed, kind=kind, holes_permille=holes, relief=relief, nodata=NODATA, out=self.dem)

    def step(self):
        self.dev.flow_routing(self.dem, NODATA, out_fdr=self.fdr, out_fac=self.fac)  # one C-ABI call

    def violations(self):
        return self.dev.check_accumulation(self.fdr, self.fac)

    def max_fac(self):
        return int(self.fac.max().item())

    def strip_checksums(self, bounds):
        return [(checksum(self.torch, self.fdr[r0:r1], r0, self.S), checksum(self.torch, self.fac[r0:r1], r0, self.S))
                for r0, r1 in bounds]


def windows_vs_oracle(torch, np, oracle, fdr_rows, row0, n_rows, total, gen, wins):
    """Direction codes of the windows `wins` [(global row, col, height, width)] of this rank's rows
    [row0, row0 + n_rows) against the CPU oracle run on the HOST-generated DEM of the window plus its ring (rows and
    columns outside the raster are nodata): independent of whatever travelled between the GPUs."""
    ok = True
    for (r, c, h, w) in wins:
        r_lo, r_hi = max(r, row0), min(r + h, row0 + n_rows)
        if r_hi <= r_lo:
            continue
        c_hi = min(c + w, total)
        pad = np.full((r_hi - r_lo + 2, c_hi - c + 2), NODATA, dtype=np.float32)
        g_r0, g_c0 = max(r_lo - 1, 0), max(c - 1, 0)
        g_r1, g_c1 = min(r_hi + 1, total), min(c_hi + 1, total)
        pad[g_r0 - (r_lo - 1) : g_r1 - (r_lo - 1), g_c0 - (c - 1) : g_c1 - (c - 1)] = gen(g_r0, g_c0, g_r1 - g_r0, g_c1 - g_c0)
        want = oracle.flow_direction_for_tile(pad, NODATA)[1:-1, 1:-1]
        got = fdr_rows[r_lo - row0 : r_hi - row0, c:c_hi].cpu().numpy()
        ok &= bool(np.array_equal(got, want))
    return ok


def run_native(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from overflow_b200 import _native, device as dev, strips

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torchrun (one rank per GPU)")
    numa = bind_to_gpu_numa(local) if (world > 1 and not args.no_numa) else None
    torch.cuda.set_device(local)
    _native.init(local)
    if world > 1:
        # NCCL announces its version on stdout when the first communicator comes up; stdout carries exactly
        # one JSON line, so that goes to stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    S = args.size
    peak, peak_src = measured_hbm_peak()
    cells_total = S * S
    bounds = strips.partition_rows(S, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allsum(v):
        if world == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    def allmax(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if world > 1:
        runner = strips.StripPipeline(S, S, rank, world, nodata=NODATA, device=torch.device("cuda", local))
        load = lambda seed, kind, holes, relief=1000.0: runner.load_synthetic(seed=seed, kind=kind, holes_permille=holes, relief=relief)  # noqa: E731
        step = runner.step
        violations = lambda: allsum(runner.check())  # noqa: E731
        max_fac = lambda: int(allmax(float(runner.fac.max().item())))  # noqa: E731
        my_fdr, my_fac = (lambda: runner.fdr), (lambda: runner.fac)
    else:
        runner = SingleRunner(torch, dev, S)
        load, step, violations, max_fac = runner.load, runner.step, runner.violations, runner.max_fac
        my_fdr, my_fac = (lambda: runner.fdr), (lambda: runner.fac)
    r0, r1 = bounds[rank]

    def timed(n_steps, n_warm):
        """(ms per step [max over ranks], phases ms per step [this rank], launches [all ranks], clocks)"""
        for _ in range(n_warm):
            step()
        barrier()
        _native.phase_timing_read(reset=True)
        _native.phase_timing_enable(True)
        _native.launch_count_reset()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clocks:
            barrier()
            ev0.record()
            for _ in range(n_steps):
                step()
            ev1.record()
            barrier()
        ms = allmax(ev0.elapsed_time(ev1))
        launches = allsum(_native.launch_count())
        _native.phase_timing_enable(False)
        phases = _native.phase_timing_read(reset=True)
        return ms / n_steps, {k: v[0] / n_steps for k, v in phases.items()}, launches, clocks.summary()

    # ---- the single-GPU run of the whole raster the strips are compared with (N > 1; rank 0 computes it)
    single = {"runner": None, "size": None}

    def equal_single_gpu(size, seed, kind, holes, relief, fdr_t, fac_t, row0, part):
        """Every strip's (fdr, fac) checksums == the same rows of a 1-GPU run of the same raster.  True / False."""
        if world == 1:
            return None
        exp = torch.zeros((world, 2), dtype=torch.int64, device="cuda")
        if rank == 0:
            if single["size"] != size:
                single["runner"] = None
                torch.cuda.empty_cache()
                single["runner"], single["size"] = SingleRunner(torch, dev, size), size
            sr = single["runner"]
            sr.load(seed, kind, holes, relief)
            sr.step()
            bad = sr.violations()
            sums = sr.strip_checksums(part)
            exp = torch.tensor(sums, dtype=torch.int64, device="cuda")
            if bad:
                exp += 1  # a single-GPU result that fails its own check must not certify anything
        dist.broadcast(exp, src=0)
        mine = (checksum(torch, fdr_t, row0, size), checksum(torch, fac_t, row0, size))
        same = int(mine[0] == int(exp[rank, 0].item()) and mine[1] == int(exp[rank, 1].item()))
        return allsum(same) == world

    def boundary_windows(size, part, rnk):
        """Windows (row, col, h, w) of rank `rnk`: the first and last rows of its strip (the rows whose codes depend
        on the neighbour's halo row) plus, on one GPU, a few random interior windows."""
        wsz = min(384, size - 2)
        a, b = part[rnk]
        rng = np.random.default_rng(1000 + rnk)
        cols = [0, size - wsz] + [int(rng.integers(0, size - wsz + 1)) for _ in range(2)]
        wins = [(a, cols[0], min(wsz, b - a), wsz), (max(a, b - wsz), cols[1], min(wsz, b - a), wsz)]
        if len(part) > 1:
            wins += [(a, cols[2], min(64, b - a), wsz), (max(a, b - 64), cols[3], min(64, b - a), wsz)]
        else:
            wins += [(int(rng.integers(0, size - wsz + 1)), cols[2], wsz, wsz), (int(rng.integers(0, size - wsz + 1)), cols[3], wsz, wsz)]
        return wins

    def parity_block(size, part, seed, kind, holes, relief, fdr_t, fac_t, row0, viol, mfac):
        import oracle

        gen = lambda gr, gc, nr, nc: oracle.synth_dem(nr, nc, row0=gr, col0=gc, total_rows=size, total_cols=size, seed=seed,  # noqa: E731
                                                      kind=kind, relief=relief, holes_permille=holes, nodata=NODATA)
        ok = windows_vs_oracle(torch, np, oracle, fdr_t, row0, fdr_t.shape[0], size, gen, boundary_windows(size, part, rank))
        ok = allsum(int(ok)) == world
        return {"accumulation_recurrence_violations": viol, "strips_equal_single_gpu": equal_single_gpu(
                    size, seed, kind, holes, relief, fdr_t, fac_t, row0, part),
                "direction_windows_vs_oracle": ok, "windows": 4 * world, "max_fac": mfac}

    # ================================================================ the headline workload
    load(args.seed, args.kind, args.holes)
    ms_per_step, per_step, launches, clocks = timed(args.steps, args.warmup)
    value = cells_total / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs:  # before anything below overwrites the step's buffers

        def sum_ranks(a):
            t = torch.from_numpy(a).cuda()
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return t.cpu().numpy()

        dump_outputs(args.dump_outputs if rank == 0 else None, my_fdr(), my_fac(), r0, S, S,
                     sum_ranks if world > 1 else None)

    # ---- roofline (live CUDA-event times from the timed region, this rank).  SURVEY 8(d) states the algorithmic
    #      bytes per stage: direction 5 B/cell, accumulation 9 B/cell (1 B code read + 8 B count write).  The
    #      accumulation stage is three kernels -- tile pass A, the perimeter-graph solve, the final tile pass --
    #      so its launch time is the sum of theirs; `kernels` also gives every kernel on its own share of those
    #      bytes (pass A: the 1 B code read, final pass: the 8 B count write).
    cells_rank = cells_total // world
    acc_ms = per_step["acc_tile_a"] + per_step["acc_solve"] + per_step["acc_tile_b"] + per_step["strip_edge"]
    stage_ms = {"flow_direction": per_step["direction"], "flow_accumulation": acc_ms}
    stage_bytes = {"flow_direction": DIR_BYTES_PER_CELL, "flow_accumulation": ACC_BYTES_PER_CELL}
    stage_kernels = {"flow_direction": "direction_kernel",
                     "flow_accumulation": "acc_tile_kernel + pj_solve_kernel (perimeter-graph solve) + acc_final_kernel"}

    def gbs(bytes_per_cell, ms_):
        return cells_rank * bytes_per_cell / (ms_ * 1e-3) / 1e9 if ms_ > 0 else None

    dom = max(stage_ms, key=stage_ms.get)
    achieved = gbs(stage_bytes[dom], stage_ms[dom]) or 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("rows") == S and tj.get("cols") == S and world == 1:
            keys = ["direction"] if dom == "flow_direction" else ["acc_tile_a", "acc_solve", "acc_tile_b"]
            traffic = float(sum(tj.get(k, 0.0) for k in keys))
    except Exception:
        pass
    kernel_ms = sum(per_step[k] for k in ("direction", "acc_tile_a", "acc_solve", "acc_tile_b", "strip_edge"))
    roofline = {
        "bound": "hbm", "kernel": f"{dom}: {stage_kernels[dom]}", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "bytes_per_cell": stage_bytes[dom],
        "avg_launch_ms": stage_ms[dom],
        # SURVEY 8(d): both denominators -- `peak` is the measured copy bandwidth, this one the nominal HBM3e figure
        "peak_nominal": HBM_NOMINAL_GBS, "frac_of_nominal": achieved / HBM_NOMINAL_GBS,
        "phases_ms_per_step": {k: round(v, 4) for k, v in per_step.items()},
        "exchange_and_host_ms": round(ms_per_step - kernel_ms, 4),
        "stages": {k: {"ms": stage_ms[k], "bytes_per_cell": stage_bytes[k], "gbs": gbs(stage_bytes[k], stage_ms[k]),
                       "frac": (gbs(stage_bytes[k], stage_ms[k]) or 0.0) / peak} for k in stage_ms},
        "kernels": {k: {"ms": per_step[k], "bytes_per_cell": PHASE_BYTES[k], "gbs": gbs(PHASE_BYTES[k], per_step[k]),
                        "frac": (gbs(PHASE_BYTES[k], per_step[k]) or 0.0) / peak} for k in PHASE_BYTES},
        "whole_step_13B_per_cell": {"ms": ms_per_step, "gbs": gbs(13.0, ms_per_step),
                                    "frac": (gbs(13.0, ms_per_step) or 0.0) / peak},
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32->u8->int64", "data": "synthetic", "config": workload_config(args, world),
        "clocks": clocks, "gpu_launches": launches, "roofline": roofline,
    }

    # ---- parity on the benchmarked result (outside the timed region), at every N
    if not args.no_check:
        line["parity"] = parity_block(S, bounds, args.seed, args.kind, args.holes, 1000.0, my_fdr(), my_fac(), r0,
                                      violations(), max_fac())

    # ---- BASELINE.json configs[3] / configs[4]: the flat-heavy and the adversarial long-path DEMs, same step, same
    #      checks (outside the headline's timed region)
    if not args.no_other:
        others = {}
        for name, size, kind, holes, relief, note in (
            ("terraced_16k", min(S, 16384), 1, 50, 200.0, "config 4: 1 m terraces (large flats, code 8), 5 % nodata holes"),
            ("tilted_plane", S, 2, 0, 1000.0, "config 5(i): every column one chain of `rows` cells through all strips"),
            ("serpentine", S, 3, 0, 1000.0, "config 5(ii): ONE channel of ~rows*cols/2 cells through every tile (east-west "
                                            "runs, stepping down at the ends), walls draining into it, a single interior "
                                            "outlet; the perimeter graph is one chain of 33 million nodes at 64k"),
            ("serpentine_ns", S, 4, 0, 1000.0, "config 5(ii) transposed: the channel runs north-south and crosses every "
                                               "row-strip boundary cols/2 times (the strip-boundary forest is one chain)"),
        ):
            if size == S:
                load(args.seed, kind, holes, relief)
                o_ms, o_ph, _, _ = timed(3, 1)
                part, fdr_t, fac_t, row0 = bounds, my_fdr(), my_fac(), r0
                viol, mfac = violations(), max_fac()
            elif world > 1:
                small = strips.StripPipeline(size, size, rank, world, nodata=NODATA, device=torch.device("cuda", local))
                small.load_synthetic(seed=args.seed, kind=kind, holes_permille=holes, relief=relief)
                saved_step, step = step, small.step
                o_ms, o_ph, _, _ = timed(3, 1)
                step = saved_step
                part = strips.partition_rows(size, world)
                fdr_t, fac_t, row0 = small.fdr, small.fac, part[rank][0]
                viol, mfac = allsum(small.check()), int(allmax(float(small.fac.max().item())))
            else:
                small = SingleRunner(torch, dev, size)
                small.load(args.seed, kind, holes, relief)
                saved_step, step = step, small.step
                o_ms, o_ph, _, _ = timed(3, 1)
                step = saved_step
                part, fdr_t, fac_t, row0 = [(0, size)], small.fdr, small.fac, 0
                viol, mfac = small.violations(), small.max_fac()
            entry = {
                "workload": f"synthetic {size}x{size} float32 DEM ({KINDS[kind]}, {holes} permille nodata holes)", "note": note,
                "ms_per_step": o_ms, "value": size * size / (o_ms * 1e-3) / 1e9, "unit": UNIT,
                "phases_ms_per_step": {k: round(v, 4) for k, v in o_ph.items() if v > 0},
                "undefined_or_nodata_fraction": float(allsum(int((fdr_t >= 8).sum().item())) / (size * size)),
            }
            if not args.no_check:
                entry["parity"] = parity_block(size, part, args.seed, kind, holes, relief, fdr_t, fac_t, row0, viol, mfac)
            others[name] = entry
            small = fdr_t = fac_t = None
        line["other_workloads"] = others
        load(args.seed, args.kind, args.holes)  # the legs below run on the headline DEM again
        step()
    single["runner"] = None
    torch.cuda.empty_cache()

    # ---- CPU baseline: the oracle port on a bounded sample of the same DEM (rank 0, N=1 only)
    if world == 1 and not args.no_cpu:
        import oracle

        sample = min(S, args.cpu_sample)
        dem_pad = np.full((sample + 2, sample + 2), NODATA, dtype=np.float32)
        dem_pad[1:-1, 1:-1] = runner.dem[:sample, :sample].cpu().numpy()
        cpu_pass(oracle, dem_pad[:66, :66])  # warm-up (thread pool)
        best = None
        for _ in range(2):
            _, _, td, ta = cpu_pass(oracle, dem_pad)
            if best is None or td + ta < best[0] + best[1]:
                best = (td, ta)
        line["cpu_baseline"] = {
            "value": sample * sample / (best[0] + best[1]) / 1e9, "unit": UNIT, "cores": oracle.num_threads(),
            "kind": "port",
            "sample": f"{sample}x{sample} window of the benchmark DEM; direction {best[0] * 1e3:.0f} ms on "
                      f"{oracle.num_threads()} threads, accumulation {best[1] * 1e3:.0f} ms on 1 thread (serial algorithm)",
        }

    # ---- SURVEY 8(f) rows, reported next to the headline
    if world == 1 and not args.no_flats:
        line["next_rows"] = {"fix_flats": flats_leg(torch, dev, peak), "breach_single_cell_pits": pits_leg(torch, dev, peak)}

    # ---- end to end through the public host API: pinned host buffers, H2D + D2H inside the timed region
    if world == 1 and not args.no_e2e:
        from overflow_b200.flow_routing import flow_routing_for_raster

        h_dem = torch.empty((S, S), dtype=torch.float32, pin_memory=True)
        h_dem.copy_(runner.dem)
        runner.dem = runner.fdr = runner.fac = None  # the host API stages through the library's own buffers
        torch.cuda.empty_cache()
        h_fdr = torch.empty((S, S), dtype=torch.uint8, pin_memory=True)
        h_fac = torch.empty((S, S), dtype=torch.int64, pin_memory=True)
        n_dem, n_fdr, n_fac = h_dem.numpy(), h_fdr.numpy(), h_fac.numpy()

        def e2e_step():
            flow_routing_for_raster(n_dem, NODATA, out_fdr=n_fdr, out_fac=n_fac)

        e2e_step()  # warm-up: allocates the library's device staging
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        el = (time.perf_counter() - t0) / args.e2e_steps
        line["e2e"] = {
            "value": cells_total / el / 1e9, "unit": UNIT,
            "h2d_bytes_per_step": int(cells_total * 4), "d2h_bytes_per_step": int(cells_total + cells_total * 8),
            "ms_per_step": el * 1e3, "steps": args.e2e_steps,
            "api": "overflow_b200.flow_routing.flow_routing_for_raster (C ABI ofl_flow_routing_f32, OFL_MEM_HOST) on pinned "
                   "host arrays: DEM in, codes and counts out",
        }
    elif world > 1 and not args.no_e2e:
        # every rank streams its strip from / to pinned host memory around the distributed step
        h_dem = torch.empty(tuple(runner.dem.shape), dtype=torch.float32, pin_memory=True)
        h_dem.copy_(runner.dem)
        h_fdr = torch.empty(tuple(runner.fdr.shape), dtype=torch.uint8, pin_memory=True)
        h_fac = torch.empty(tuple(runner.fac.shape), dtype=torch.int64, pin_memory=True)
        copy_stream = torch.cuda.Stream()
        ev_codes = torch.cuda.Event()

        # the PCIe ceiling of this box with all ranks copying at once (no compute): the strip up, then codes + counts down
        def copies_only():
            runner.dem.copy_(h_dem, non_blocking=True)
            h_fdr.copy_(runner.fdr, non_blocking=True)
            h_fac.copy_(runner.fac, non_blocking=True)
            torch.cuda.synchronize()

        copies_only()
        barrier()
        t0 = time.perf_counter()
        copies_only()
        barrier()
        ceiling_s = allmax(time.perf_counter() - t0)

        # ... and with the two directions at once (PCIe is full duplex): what overlapping one step's download with the
        # next step's upload could reach at best -- the step itself cannot (the counts need every code)
        def copies_duplex():
            with torch.cuda.stream(copy_stream):
                runner.dem.copy_(h_dem, non_blocking=True)
            h_fdr.copy_(runner.fdr, non_blocking=True)
            h_fac.copy_(runner.fac, non_blocking=True)
            torch.cuda.synchronize()

        copies_duplex()
        barrier()
        t0 = time.perf_counter()
        copies_duplex()
        barrier()
        duplex_s = allmax(time.perf_counter() - t0)

        def e2e_step():
            cur = torch.cuda.current_stream()
            runner.dem.copy_(h_dem, non_blocking=True)
            runner.fill_edge_halos()
            runner._exchange_halo(runner.dem_halo)
            runner.direction()
            ev_codes.record(cur)
            with torch.cuda.stream(copy_stream):  # the codes go home while the accumulation runs
                copy_stream.wait_event(ev_codes)
                h_fdr.copy_(runner.fdr, non_blocking=True)
            runner._exchange_halo(runner.fdr_halo)
            runner.accum_local()
            dist.all_gather_into_tensor(runner.rec_all, runner.rec)
            runner.boundary_solve()
            runner.accum_final()
            h_fac.copy_(runner.fac, non_blocking=True)
            runner.collect_flags()
            dist.all_reduce(runner.flags, op=dist.ReduceOp.MAX)
            strips.raise_for_flags(runner.flags.tolist())
            torch.cuda.synchronize()

        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        barrier()
        el = allmax((time.perf_counter() - t0) / args.e2e_steps)
        bytes_step = cells_total * 13
        line["e2e"] = {
            "value": cells_total / el / 1e9, "unit": UNIT,
            "h2d_bytes_per_step": int(cells_total * 4), "d2h_bytes_per_step": int(cells_total * 9),
            "ms_per_step": el * 1e3, "steps": args.e2e_steps,
            "host_copy_GBps": bytes_step / el / 1e9,
            "copies_only_ms": ceiling_s * 1e3, "copies_only_GBps": bytes_step / ceiling_s / 1e9,
            "copies_duplex_ms": duplex_s * 1e3, "copies_duplex_GBps": bytes_step / duplex_s / 1e9,
            "fraction_of_copy_ceiling": ceiling_s / el,
            "copies_only_note": "the same pinned copies with no kernels and no NCCL, all ranks at once: what the box's "
                                "PCIe / host memory gives this transfer pattern",
            "host_binding": numa or "none",
            "api": "per rank: pinned host strip -> device, StripPipeline phases (the codes leave for the host while the "
                   "accumulation runs), counts -> pinned host",
        }

    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def flats_leg(torch, dev, peak, size=8192, window=1024):
    """ofl_fix_flats_f32 (resolve_flats + d8_masked_flow_dirs) on device buffers: terraced synthetic DEM, CUDA-event
    time of the call, a window checked against the CPU oracle, and the oracle timed on that window."""
    import numpy as np

    import oracle

    dem = dev.synth_dem(size, size, seed=3, kind=1, relief=200.0, holes_permille=5)
    fdr0 = dev.flow_direction(dem, NODATA).contiguous()
    work = dev.flats_workspace(size, size)
    flat_mask = torch.empty((size, size), dtype=torch.int32, device="cuda")
    labels = torch.empty((size, size), dtype=torch.int32, device="cuda")
    fdr = fdr0.clone()
    times, info = [], None
    for it in range(4):
        fdr.copy_(fdr0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _, info = dev.fix_flats(dem, fdr, workspace=work, flat_mask=flat_mask, labels=labels)
        e1.record()
        torch.cuda.synchronize()
        if it:
            times.append(e0.elapsed_time(e1))
    ms = float(np.median(times))
    cells = size * size
    hd, hf = dem[:window, :window].contiguous().cpu().numpy(), fdr0[:window, :window].contiguous().cpu().numpy()
    t0 = time.perf_counter()
    want_mask, want_labels = oracle.resolve_flats(hd, hf)
    want = oracle.d8_masked_flow_dirs(want_mask, hf, want_labels)
    cpu_s = time.perf_counter() - t0
    got = dev.fix_flats(torch.from_numpy(hd).cuda(), torch.from_numpy(hf).cuda())[0].cpu().numpy()
    return {
        "api": "ofl_fix_flats_f32 on device buffers (reference fix_flats.py: resolve_flats + d8_masked_flow_dirs)",
        "workload": f"synthetic {size}x{size} terraced float32 DEM (1 m steps, 5 permille nodata holes, seed 3)",
        "ms": ms, "value": cells / ms / 1e6, "unit": UNIT,
        "cells_without_direction": int((fdr0 == 8).sum().item()), "left_without_direction": int((fdr == 8).sum().item()),
        "flats": info[2], "sweep_levels": [info[3], info[4]],
        "roofline": {"bound": "hbm", "bytes_per_cell": 14.0, "achieved": cells * 14.0 / ms / 1e6, "peak": peak,
                     "unit": "GB/s", "frac": cells * 14.0 / ms / 1e6 / peak,
                     "note": "graph work (union-find + breadth-first sweeps): bound by dependent scattered accesses, not by streaming"},
        "parity": {"window": window, "codes_equal_oracle": bool(np.array_equal(got, want))},
        "cpu_baseline": {"value": window * window / cpu_s / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": f"{window}x{window} window of the same DEM (the reference algorithm is serial)"},
    }


def pits_leg(torch, dev, peak, size=16384, window=2048):
    """ofl_breach_single_cell_pits_f32 on device buffers: fractal synthetic DEM, CUDA-event time of the call, a window
    breached on its own and compared with the CPU oracle, and the oracle timed on that window."""
    import numpy as np

    import oracle

    dem0 = dev.synth_dem(size, size, seed=3, kind=0, holes_permille=5)
    dem = dem0.clone()
    times, info = [], None
    for it in range(4):
        dem.copy_(dem0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _, info = dev.breach_single_cell_pits(dem, NODATA)
        e1.record()
        torch.cuda.synchronize()
        if it:
            times.append(e0.elapsed_time(e1))
    ms = float(np.median(times))
    cells = size * size
    hw = dem0[:window, :window].contiguous().cpu().numpy()
    t0 = time.perf_counter()
    want, want_unsolved = oracle.breach_single_cell_pits_in_chunk(hw, NODATA)
    cpu_s = time.perf_counter() - t0
    d_w = torch.from_numpy(hw.copy()).cuda()
    got_unsolved, _ = dev.breach_single_cell_pits(d_w, NODATA)
    ok = bool(np.array_equal(d_w.cpu().numpy().view(np.uint32), want.view(np.uint32))
              and np.array_equal(got_unsolved.cpu().numpy(), want_unsolved))
    return {
        "api": "ofl_breach_single_cell_pits_f32 on device buffers (reference breach_single_cell_pits_in_chunk)",
        "workload": f"synthetic {size}x{size} float32 DEM (fractal value-noise, 5 permille nodata holes, seed 3)",
        "ms": ms, "value": cells / ms / 1e6, "unit": UNIT, "pits": info[0], "unsolved": info[1], "rounds": info[2],
        "roofline": {"bound": "hbm", "bytes_per_cell": 5.0, "achieved": cells * 5.0 / ms / 1e6, "peak": peak, "unit": "GB/s",
                     "frac": cells * 5.0 / ms / 1e6 / peak,
                     "note": "4 B DEM read + 1 B unsolved raster written per cell; breached cells (about 1 %) are rewritten in place"},
        "parity": {"window": window, "bits_equal_oracle": ok},
        "cpu_baseline": {"value": window * window / cpu_s / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": f"{window}x{window} window of the same DEM (the reference's second pass is serial)"},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--size", type=int, default=65536)
    ap.add_argument("--kind", type=int, default=0)
    ap.add_argument("--holes", type=int, default=5, help="nodata holes, permille of the raster")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=8192)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-other", action="store_true", help="skip the flat-heavy / long-path workloads")
    ap.add_argument("--no-flats", action="store_true", help="skip the fix_flats / pit breaching legs (next_rows)")
    ap.add_argument("--no-numa", action="store_true", help="N > 1: do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-numba", action="store_true", help="reference arm: C port for direction even if oracle/_ref exists")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the codes and counts of the last timed step (a fixed sample of cells of a large raster) "
                         "as DIR/fdr.npy, DIR/fac.npy and their cell indices as DIR/cells.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
