"""GPU: drainage-basin labelling through the C ABI against the serial CPU reference, the outlet-size identity with
the accumulation, cycles, the checker, workspace sizing and the file driver / CLI."""
import click.testing
import numpy as np
import pytest

import basins_reference as ref
import oracle
from oracle import synth
from conftest import load_golden
from test_oracle import ACC_CASES

pytestmark = pytest.mark.gpu


def codes_of(dem):
    return np.ascontiguousarray(oracle.flow_direction_for_tile(synth.pad_nodata(dem), synth.NODATA)[1:-1, 1:-1])


def device_codes(rows, cols, kind, seed=0, holes_permille=0):
    from overflow_b200 import device as dev

    return dev.flow_direction(dev.synth_dem(rows, cols, seed=seed, kind=kind, holes_permille=holes_permille),
                              synth.NODATA)


def host_and_device(fdr, pour_points=None):
    """Labels through the host API and the device API (same result required); returns the host result."""
    import torch

    from overflow_b200 import device as dev
    from overflow_b200.basins import label_basins

    got = label_basins(fdr, pour_points)
    got_dev = dev.label_basins(torch.from_numpy(np.ascontiguousarray(fdr, dtype=np.uint8)).cuda(),
                               pour_points=pour_points)
    assert np.array_equal(got_dev.cpu().numpy(), got)
    return got


def test_kat():
    fdr = load_golden("kat.npz")["acc_fdr"]
    assert np.array_equal(host_and_device(fdr), ref.basins(fdr))


@pytest.mark.parametrize("name", ACC_CASES)
def test_golden_codes(name):
    fdr = load_golden("accumulation.npz")[f"{name}_fdr"]
    assert np.array_equal(host_and_device(fdr), ref.basins(fdr))


def _fuzzed():
    fdr = codes_of(synth.fractal(300, 400, beta=2.0, seed=11))
    rng = np.random.default_rng(12)
    idx = rng.random(fdr.shape) < 0.05  # codes after the stencil: removing edges cannot close a cycle
    fdr[idx] = rng.choice(np.array([8, 9, 10, 11, 100, 254, 255], dtype=np.uint8), size=int(idx.sum()))
    return fdr


def _cases():
    yield "fractal_holes_700x900", lambda: codes_of(synth.punch_holes(synth.fractal(700, 900, beta=2.0, seed=0),
                                                                     frac=0.01, seed=1))
    yield "terraced", lambda: codes_of(synth.terraced(600, 800, seed=4))
    yield "tilted", lambda: codes_of(synth.tilted_plane(900, 300))
    yield "serpentine_kind3", lambda: device_codes(320, 520, 3).cpu().numpy()
    yield "serpentine_kind4", lambda: device_codes(520, 320, 4).cpu().numpy()
    yield "fuzzed", _fuzzed
    yield "random_acyclic", lambda: ref.random_acyclic_codes(150, 170, seed=5)


@pytest.mark.parametrize("name,make", list(_cases()), ids=[n for n, _ in _cases()])
def test_vs_reference(name, make):
    fdr = make()
    if name == "terraced":
        assert (fdr == 8).sum() > 1000
    assert np.array_equal(host_and_device(fdr), ref.basins(fdr))


@pytest.mark.parametrize("shape", [(1, 4097), (4097, 1), (63, 65), (65, 63), (64, 64), (129, 4097)])
def test_shapes(shape):
    fdr = codes_of(synth.fractal(*shape, beta=2.0, seed=sum(shape)))
    assert np.array_equal(host_and_device(fdr), ref.basins(fdr))


def test_padded_device_tensors():
    import torch

    from overflow_b200 import device as dev

    fdr = codes_of(synth.punch_holes(synth.fractal(333, 250, beta=2.0, seed=3), frac=0.02, seed=4))
    want = ref.basins(fdr)
    buf = torch.full((333, 320), 7, dtype=torch.uint8, device="cuda")
    d_fdr = buf[:, :250]
    d_fdr.copy_(torch.from_numpy(fdr))
    out_buf = torch.full((333, 262), -5, dtype=torch.int64, device="cuda")
    out = out_buf[:, :250]
    got = dev.label_basins(d_fdr, out=out, workspace=dev.basins_workspace(333, 250))
    assert got.data_ptr() == out.data_ptr()
    assert np.array_equal(out.cpu().numpy(), want)
    assert (out_buf[:, 250:] == -5).all()  # nothing written past the raster's columns
    assert dev.check_basins(d_fdr, out) == 0


def _pour_points(fdr, seed, k=25):
    rows, cols = fdr.shape
    rng = np.random.default_rng(seed)
    pp = np.stack([rng.integers(0, rows, k), rng.integers(0, cols, k)], axis=1)
    succ = ref.successors(fdr)
    nested = []
    for r, c in pp[:5]:  # a pour point a few steps downstream of another one
        i = r * cols + c
        for _ in range(7):
            if succ[i] >= 0:
                i = succ[i]
        nested.append(divmod(int(i), cols))
    nodata = np.argwhere(fdr == 9)[:2]
    outlet = np.argwhere(((succ < 0) & (fdr.reshape(-1) != 9)).reshape(rows, cols))[:2]
    return np.vstack([pp, np.array(nested), nodata, pp[:3], outlet]).astype(np.int64)


@pytest.mark.parametrize("seed", [0, 1])
def test_pour_points(seed):
    fdr = codes_of(synth.punch_holes(synth.fractal(400, 530, beta=2.0, seed=20 + seed), frac=0.01, seed=2))
    pp = _pour_points(fdr, seed)
    want = ref.basins(fdr, pp)
    got = host_and_device(fdr, pp)
    assert np.array_equal(got, want)
    assert len(np.unique(want)) > 10
    from overflow_b200.basins import check_basins

    assert check_basins(fdr, got, pp) == 0


def test_pour_point_outside_raster_through_the_abi():
    import torch

    from overflow_b200 import _native, device as dev

    fdr = torch.full((70, 80), 8, dtype=torch.uint8, device="cuda")
    out = torch.empty((70, 80), dtype=torch.int64, device="cuda")
    ws = dev.basins_workspace(70, 80)
    pour = torch.tensor([5, 70 * 80], dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    rc = _native.lib().ofl_label_basins_u8(fdr.data_ptr(), 70, 80, 80, pour.data_ptr(), 2, out.data_ptr(), 80,
                                           ws.data_ptr(), ws.numel(), _native.OFL_MEM_DEVICE, None)
    assert rc == _native.OFL_ERR_INVALID


def _outlet_sizes_match(fdr):
    import torch

    from overflow_b200 import device as dev

    labels = dev.label_basins(fdr)
    fac = dev.flow_accumulation(fdr)
    assert dev.check_basins(fdr, labels) == 0
    flat = labels.reshape(-1)
    n = flat.numel()
    idx = torch.arange(n, device=flat.device, dtype=torch.int64)
    outlet = flat == idx + 1
    counts = torch.bincount(flat, minlength=n + 1)
    assert int(outlet.sum()) > 0
    assert torch.equal(counts[idx[outlet] + 1], fac.reshape(-1)[outlet])
    assert int(counts[1:].sum()) == int((fdr != 9).sum())  # every data cell reaches an outlet


def test_outlet_sizes_fractal_4096():
    _outlet_sizes_match(device_codes(4096, 4096, 0, seed=9, holes_permille=5))


def test_outlet_sizes_serpentine_2048():
    _outlet_sizes_match(device_codes(2048, 2048, 3))


@pytest.mark.parametrize("cells", [((10, 10), (10, 11)), ((20, 63), (20, 64)), ((63, 30), (64, 30))],
                         ids=["in_tile", "cols_63_64", "rows_63_64"])
def test_cycle_is_reported(cells):
    import torch

    from overflow_b200 import _native, device as dev
    from overflow_b200.basins import label_basins

    fdr = np.full((130, 140), 8, dtype=np.uint8)
    (r0, c0), (r1, c1) = cells
    if r0 == r1:
        fdr[r0, c0], fdr[r1, c1] = 0, 4  # east / west
    else:
        fdr[r0, c0], fdr[r1, c1] = 6, 2  # south / north
    fdr[r0, c0 - 1] = 0  # a cell upstream of the cycle
    with pytest.raises(_native.OverflowB200Error) as e:
        label_basins(fdr)
    assert e.value.status == _native.OFL_ERR_CYCLE
    with pytest.raises(_native.OverflowB200Error) as e:
        dev.label_basins(torch.from_numpy(fdr).cuda())
    assert e.value.status == _native.OFL_ERR_CYCLE
    ok = codes_of(synth.fractal(130, 140, beta=2.0, seed=1))
    assert np.array_equal(host_and_device(ok), ref.basins(ok))


def _violations(fdr, labels, pour_points=None):
    """numpy restatement of the checker's rule."""
    rows, cols = fdr.shape
    flat = labels.reshape(-1)
    code = fdr.reshape(-1)
    succ = ref.successors(fdr)
    is_pour = np.zeros(rows * cols, dtype=bool)
    if pour_points is not None:
        is_pour[np.asarray(pour_points)[:, 0] * cols + np.asarray(pour_points)[:, 1]] = True
    own = np.arange(1, rows * cols + 1)
    want = np.where(is_pour | (pour_points is None), own, 0)
    follow = (succ >= 0) & ~is_pour
    want = np.where(follow, flat[np.maximum(succ, 0)], want)
    want = np.where(code == 9, 0, want)
    return int((flat != want).sum())


@pytest.mark.parametrize("with_pour", [False, True])
def test_checker(with_pour):
    from overflow_b200.basins import check_basins

    fdr = codes_of(synth.punch_holes(synth.fractal(300, 333, beta=2.5, seed=12), frac=0.01, seed=3))
    pp = _pour_points(fdr, 4) if with_pour else None
    labels = ref.basins(fdr, pp)
    assert check_basins(fdr, labels, pp) == 0 == _violations(fdr, labels, pp)
    rng = np.random.default_rng(5)
    for _ in range(5):
        bad = labels.copy()
        r, c = rng.integers(0, 300), rng.integers(0, 333)
        bad[r, c] += 1
        n = check_basins(fdr, bad, pp)
        assert n == _violations(fdr, bad, pp) >= 1


def test_checker_16384_fractal():
    from overflow_b200 import device as dev

    fdr = device_codes(16384, 16384, 0, seed=4, holes_permille=3)
    labels = dev.label_basins(fdr)
    assert dev.check_basins(fdr, labels) == 0


def test_workspace_one_byte_short():
    import torch

    from overflow_b200 import _native, device as dev

    rows, cols = 200, 300
    fdr = torch.full((rows, 304), 8, dtype=torch.uint8, device="cuda")[:, :cols]
    out = torch.empty((rows, cols), dtype=torch.int64, device="cuda")
    need = int(_native.lib().ofl_basins_workspace_bytes(rows, cols))
    ws = torch.empty((need,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    rc = _native.lib().ofl_label_basins_u8(fdr.data_ptr(), rows, cols, 304, None, 0, out.data_ptr(), cols,
                                           ws.data_ptr(), need - 1, _native.OFL_MEM_DEVICE, None)
    assert rc == _native.OFL_ERR_WORKSPACE
    rc = _native.lib().ofl_label_basins_u8(fdr.data_ptr(), rows, cols, 304, None, 0, out.data_ptr(), cols,
                                           ws.data_ptr(), need, _native.OFL_MEM_DEVICE, None)
    assert rc == 0
    want = np.arange(1, rows * cols + 1).reshape(rows, cols)  # all code 8: every cell is its own outlet
    assert np.array_equal(out.cpu().numpy(), want)


def test_phase_timing_names_the_three_passes():
    from overflow_b200 import _native
    from overflow_b200.basins import label_basins

    _native.phase_timing_enable(True)
    try:
        _native.phase_timing_read(reset=True)
        label_basins(codes_of(synth.fractal(200, 200, beta=2.0, seed=1)))
        ph = _native.phase_timing_read(reset=True)
    finally:
        _native.phase_timing_enable(False)
    for name in ("basins_tile", "basins_solve", "basins_final"):
        assert ph[name][1] >= 1


def _write_codes(path, fdr, geotransform):
    from overflow_b200.util.raster import create_raster

    ds = create_raster(path, fdr.shape[1], fdr.shape[0], "Byte", geotransform=geotransform)
    band = ds.GetRasterBand(1)
    band.WriteArray(fdr)
    band.SetNoDataValue(9)
    ds.FlushCache()


@pytest.mark.parametrize("with_pour", [False, True])
def test_file_driver_and_cli(tmp_path, with_pour):
    from overflow_b200.basins import basins, label_basins
    from overflow_b200.util.raster import open_raster
    from overflow_cli import basins_cli

    fdr = codes_of(synth.punch_holes(synth.fractal(150, 170, beta=2.0, seed=8), frac=0.02, seed=9))
    gt = (500000.0, 30.0, 0.0, 4100000.0, 0.0, -30.0)
    src = str(tmp_path / "fdr.tif")
    _write_codes(src, fdr, gt)
    pp = _pour_points(fdr, 6, k=8) if with_pour else None
    want = label_basins(fdr, pp)
    assert np.array_equal(want, ref.basins(fdr, pp))

    out = str(tmp_path / "basins.tif")
    basins(src, out, chunk_size=33, pour_points=pp)
    band = open_raster(out).GetRasterBand(1)
    assert band.GetNoDataValue() == 0
    got = band.ReadAsArray()
    assert got.dtype == np.int64 and np.array_equal(got, want)
    assert tuple(open_raster(out).GetGeoTransform()) == gt

    out_cli = str(tmp_path / "basins_cli.tif")
    args = ["--input_file", src, "--output_file", out_cli, "--chunk_size", "40"]
    if with_pour:
        pfile = tmp_path / "pour.txt"
        pfile.write_text("".join(f"{r},{c}\n" for r, c in pp))
        args += ["--pour_points", str(pfile)]
    result = click.testing.CliRunner().invoke(basins_cli, args)
    assert result.exit_code == 0, result.output
    assert np.array_equal(open_raster(out_cli).GetRasterBand(1).ReadAsArray(), want)


def test_cli_failure_exits_non_zero(tmp_path):
    from overflow_cli import basins_cli

    result = click.testing.CliRunner().invoke(
        basins_cli, ["--input_file", str(tmp_path / "missing.tif"), "--output_file", str(tmp_path / "o.tif")])
    assert result.exit_code == 1
    assert "basins failed with the following exception" in result.output

