"""bench.py prints ONE JSON line with the keys the driver reads (reference arm on CPU, native arm on a GPU)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

COMMON = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
          "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, f"stdout must be one JSON line, got {len(lines)}"
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample", "256"])
    assert d["impl"] == "reference"
    assert COMMON <= set(d)
    assert d["unit"] == "Gcells/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"].startswith("flow_direction + flow_accumulation")
    cb = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] == "port" and cb["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"]
    # the arm says what it ran, and the CUDA library is not mapped into its process
    assert d["config"]["sample_rows"] == 256 and d["config"]["rows"] == 65536
    assert all("overflow_b200" not in p for p in d["repo_libraries_loaded"])
    assert any("liboracle_d8" in p for p in d["repo_libraries_loaded"])


@pytest.mark.gpu
def test_native_arm_line():
    d = _run(["--size", "2048", "--steps", "2", "--warmup", "3", "--cpu-sample", "512"])
    assert COMMON | {"clocks", "gpu_launches", "roofline", "parity"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert d["parity"]["accumulation_recurrence_violations"] == 0 and d["parity"]["direction_windows_vs_oracle"]
    for name in ("terraced_16k", "tilted_plane", "serpentine", "serpentine_ns"):
        o = d["other_workloads"][name]
        assert o["value"] > 0 and o["parity"]["accumulation_recurrence_violations"] == 0, name
        assert o["parity"]["direction_windows_vs_oracle"], name
    assert d["other_workloads"]["serpentine"]["parity"]["max_fac"] > 2048 * 2048 // 2
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 2048 * 2048 * 4 and e["d2h_bytes_per_step"] == 2048 * 2048 * 9 and e["value"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    ff = d["next_rows"]["fix_flats"]
    assert ff["parity"]["codes_equal_oracle"] and ff["value"] > 0 and ff["left_without_direction"] < ff["cells_without_direction"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(ff["cpu_baseline"])
    bp = d["next_rows"]["breach_single_cell_pits"]
    assert bp["parity"]["bits_equal_oracle"] and bp["value"] > 0 and bp["pits"] >= bp["unsolved"] >= 0


def test_checksum_is_position_weighted_and_additive_over_strips():
    """bench.py's strip checksum: a swap of two cells changes it; strips add up to the whole raster (mod 2^64)."""
    import sys

    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    rng = np.random.default_rng(0)
    a = torch.from_numpy(rng.integers(-9998, 1 << 40, (300, 70), dtype=np.int64))
    whole = bench.checksum(torch, a, 0, 70, chunk_rows=64)
    parts = [bench.checksum(torch, a[r0:r1], r0, 70, chunk_rows=50) for r0, r1 in ((0, 128), (128, 192), (192, 300))]
    assert (sum(parts) - whole) % (1 << 64) == 0
    b = a.clone()
    b[5, 6], b[200, 3] = a[200, 3], a[5, 6]
    assert bench.checksum(torch, b, 0, 70) != whole
    c = torch.from_numpy(rng.integers(0, 10, (300, 70), dtype=np.uint8))
    assert bench.checksum(torch, c, 1000, 70) != bench.checksum(torch, c, 1001, 70)


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs on the reference arm: a window this small is written whole, codes float32 and counts float64,
    and they are the oracle's for that window of the benchmark DEM."""
    import numpy as np

    import oracle
    from oracle import synth

    _run(["--impl", "reference", "--steps", "2", "--warmup", "0", "--cpu-sample", "192", "--dump-outputs", str(tmp_path)])
    fdr, fac, cells = (np.load(tmp_path / f"{name}.npy") for name in ("fdr", "fac", "cells"))
    assert fdr.dtype == np.float32 and fac.dtype == np.float64 and cells.dtype == np.float64
    assert np.array_equal(cells, np.arange(192 * 192))
    dem = oracle.synth_dem(192, 192, total_rows=65536, total_cols=65536, seed=0, kind=0, holes_permille=5)
    want = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1]
    assert np.array_equal(fdr, want.reshape(-1))
    assert np.array_equal(fac, oracle.flow_accumulation(want).reshape(-1))


def test_dump_sample_is_fixed_and_strips_add_up_to_the_whole(tmp_path, monkeypatch):
    """The sampled cells are distinct, ascending, inside the raster and the same on every call; the three files stay
    under 64 MB; the shares of row strips (ranks of a multi-GPU run) add up to the dump of the whole raster."""
    import numpy as np

    import bench

    a = bench.dump_cells(65536, 65536)
    assert np.array_equal(a, bench.dump_cells(65536, 65536)) and len(a) == bench.DUMP_CELLS
    assert a[0] >= 0 and a[-1] < 65536 * 65536 and (np.diff(a) > 0).all()
    assert bench.DUMP_CELLS * (4 + 8 + 8) + 3 * 128 <= 64 << 20

    monkeypatch.setattr(bench, "DUMP_CELLS", 5000)
    rng = np.random.default_rng(1)
    fdr = rng.integers(0, 10, (300, 70), dtype=np.uint8)
    fac = rng.integers(-9998, 1 << 40, (300, 70), dtype=np.int64)
    bench.dump_outputs(str(tmp_path), fdr, fac, 0, 300, 70)
    whole = {name: np.load(tmp_path / f"{name}.npy") for name in ("fdr", "fac", "cells")}
    cells = whole["cells"].astype(np.int64)
    assert len(cells) == 5000
    assert np.array_equal(whole["fdr"], fdr.reshape(-1)[cells]) and np.array_equal(whole["fac"], fac.reshape(-1)[cells])
    shares = []
    for r0, r1 in ((0, 128), (128, 192), (192, 300)):
        bench.dump_outputs(None, fdr[r0:r1], fac[r0:r1], r0, 300, 70, sum_ranks=lambda s: shares.append(s) or s)
    assert np.array_equal(sum(shares[0::2]), whole["fdr"]) and np.array_equal(sum(shares[1::2]), whole["fac"])


@pytest.mark.gpu
def test_native_arm_dumps_its_last_step(tmp_path):
    """--steps sets the number of timed steps (the library's launches scale with it), and --dump-outputs writes the same
    sample on every run: the oracle's codes and counts of the benchmark DEM at those cells."""
    import numpy as np

    import oracle
    from oracle import synth

    fast = ["--size", "2048", "--warmup", "1", "--no-check", "--no-other", "--no-cpu", "--no-flats", "--no-e2e"]
    one = _run(fast + ["--steps", "1", "--dump-outputs", str(tmp_path / "one")])
    three = _run(fast + ["--steps", "3", "--dump-outputs", str(tmp_path / "three")])
    assert one["steps"] == 1 and three["steps"] == 3 and three["gpu_launches"] == 3 * one["gpu_launches"] > 0
    got = {name: np.load(tmp_path / "one" / f"{name}.npy") for name in ("fdr", "fac", "cells")}
    for name, a in got.items():
        assert np.array_equal(a, np.load(tmp_path / "three" / f"{name}.npy")), name
    assert got["fdr"].dtype == np.float32 and got["fac"].dtype == np.float64 and len(got["cells"]) == 1 << 21
    assert sum(os.path.getsize(tmp_path / "one" / f"{name}.npy") for name in got) <= 64 << 20
    dem = oracle.synth_dem(2048, 2048, seed=0, kind=0, holes_permille=5)
    want = oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1]
    cells = got["cells"].astype(np.int64)
    assert np.array_equal(got["fdr"], want.reshape(-1)[cells])
    assert np.array_equal(got["fac"], oracle.flow_accumulation(want).reshape(-1)[cells])
