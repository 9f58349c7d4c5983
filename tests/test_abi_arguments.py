"""Every compute entry point of the C ABI refuses a bad argument before it touches the device: without one the call
returns its argument status (not OFL_ERR_CUDA), and with one it launches nothing.

Each case passes buffers as large as its arguments claim: host memory where the library reads host memory, and, when
a device is present, device memory where it would read a device pointer.  Cases marked `claims_more` describe a
raster larger than the buffers they pass; they run only when neither the library nor torch finds a device, so that
a regression cannot hand them to one."""
import ctypes

import numpy as np
import pytest

from overflow_b200 import _native, build

INVALID, WORKSPACE = _native.OFL_ERR_INVALID, _native.OFL_ERR_WORKSPACE
H, D = _native.OFL_MEM_HOST, _native.OFL_MEM_DEVICE
R = C = 64  # the raster of every case that does not say otherwise
BIG = 1 << 17  # 2^34 cells as BIG x BIG / 2: beyond every whole-raster shape limit


class Buffers:
    """Keeps the buffers of one case alive and hands out their addresses."""

    def __init__(self, device):
        self.device, self.keep = device, []

    def host(self, nbytes):
        a = np.zeros(max(int(nbytes), 1), dtype=np.uint8)
        self.keep.append(a)
        return a.ctypes.data

    def dev(self, nbytes):
        """Memory the library reads as a device pointer: a CUDA tensor when a device is present."""
        if not self.device:
            return self.host(nbytes)
        import torch

        t = torch.zeros(max(int(nbytes), 1), dtype=torch.uint8, device="cuda")
        self.keep.append(t)
        return t.data_ptr()

    def mem(self, kind, nbytes):
        return self.dev(nbytes) if kind == D else self.host(nbytes)


def i64(n=1):
    return (ctypes.c_int64 * n)()


def acc(b, kind, rows=R, cols=C, ld_fdr=C, ld_fac=C, fdr=True, fac=True, work=None, n_bad=None, check=False):
    m = lambda n: b.mem(kind, n)  # noqa: E731
    f = m(rows * ld_fdr) if fdr else None
    a = m(rows * ld_fac * 8) if fac else None
    if check:
        return f, rows, cols, ld_fdr, a, ld_fac, n_bad if n_bad is not None else i64(), kind, None
    return f, rows, cols, ld_fdr, a, ld_fac, None, work, 16 if work else 0, kind, None


def flats(b, kind, rows=R, cols=C, **null):
    """Arguments of ofl_resolve_flats_f32 / ofl_fix_flats_f32; null=name makes that pointer NULL."""
    m = lambda name, n: None if null.get(name) else b.mem(kind, n)  # noqa: E731
    n = rows * cols
    work = null.get("work")
    return (m("dem", 4 * n), m("fdr", n), rows, cols, m("flat_mask", 4 * n), m("labels", 4 * n), i64(5),
            b.dev(16) if work else None, 16 if work else 0, kind, None)


def strip_local(b, rows=R, cols=C, ld=C, has_below=0, work=None):
    ws = b.dev(work if work is not None else 1 << 20)
    return (b.dev((rows + 2) * ld), rows, cols, ld, 0, has_below, b.dev(max(rows, 0) * max(cols, 0) * 8), cols, ws,
            work if work is not None else 1 << 20, b.dev(1 << 16), None)


# (id, entry point, arguments(buffers), expected status, message fragment, claims_more)
CASES = [
    ("direction_negative_rows", "ofl_flow_direction_f32",
     lambda b: (b.host(4), -3, C, C, -9999.0, b.host(1), C, 1, H, None), INVALID, "negative raster size", False),
    ("direction_unknown_mode", "ofl_flow_direction_f32",
     lambda b: (b.host(4 * R * C), R, C, C, -9999.0, b.host(R * C), C, 7, H, None), INVALID, "unknown direction mode",
     False),
    ("direction_unknown_mem_kind", "ofl_flow_direction_f32",
     lambda b: (b.host(4 * R * C), R, C, C, -9999.0, b.host(R * C), C, 1, 5, None), INVALID, "unknown mem_kind", False),
    ("direction_device_null_fdr", "ofl_flow_direction_f32",
     lambda b: (b.dev(4 * R * C), R, C, C, -9999.0, None, C, 1, D, None), INVALID, "null raster pointer", False),
    ("direction_short_ld", "ofl_flow_direction_f32",
     lambda b: (b.host(4 * R * C), R, C, C, -9999.0, b.host(R * C), C - 1, 1, H, None), INVALID, "leading dimension",
     False),
    ("direction_x64_unknown_kind", "ofl_flow_direction_x64",
     lambda b: (b.host(8 * R * C), 9, R, C, C, -9999.0, b.host(R * C), C, 1, H, None), INVALID, "unknown element kind",
     False),
    ("fill_border_negative_rows", "ofl_fill_border_u8",
     lambda b: (b.dev(1), -3, C, C, 9, None), INVALID, "negative raster size", False),
    ("fill_border_null", "ofl_fill_border_u8",
     lambda b: (None, R, C, C, 9, None), INVALID, "null raster pointer", False),
    ("fill_border_short_ld", "ofl_fill_border_u8",
     lambda b: (b.dev(R * C), R, C, C - 1, 9, None), INVALID, "leading dimension", False),
    ("accumulation_host_small_workspace", "ofl_flow_accumulation_u8",
     lambda b: acc(b, H, work=b.dev(16)), WORKSPACE, "workspace too small", False),
    ("accumulation_device_small_workspace", "ofl_flow_accumulation_u8",
     lambda b: acc(b, D, work=b.dev(16)), WORKSPACE, "workspace too small", False),
    ("accumulation_short_ld_fac", "ofl_flow_accumulation_u8",
     lambda b: acc(b, H, ld_fac=C - 1), INVALID, "leading dimension", False),
    ("accumulation_null_fac", "ofl_flow_accumulation_u8",
     lambda b: acc(b, D, fac=False), INVALID, "null raster pointer", False),
    ("accumulation_too_large", "ofl_flow_accumulation_u8",
     lambda b: (b.host(1), 1 << 30, 1, 1, b.host(8), 1, None, None, 0, H, None), INVALID, "bad raster size", True),
    ("seeded_null_fdr", "ofl_flow_accumulation_seeded_u8",
     lambda b: (None, R, C, C, b.host(8 * R * C), C, None, None, None, 0, H, None), INVALID, "null raster pointer",
     False),
    ("routing_device_null_fdr", "ofl_flow_routing_f32",
     lambda b: (b.dev(4 * R * C), R, C, C, -9999.0, None, C, b.dev(8 * R * C), C, None, D, None), INVALID,
     "null raster pointer", False),
    ("routing_host_short_ld_dem", "ofl_flow_routing_f32",
     lambda b: (b.host(4 * R * C), R, C, C - 1, -9999.0, None, C, b.host(8 * R * C), C, None, H, None), INVALID,
     "leading dimension", False),
    ("routing_host_too_large", "ofl_flow_routing_f32",
     lambda b: (b.host(4), 1 << 30, 1, 1, -9999.0, None, 1, b.host(8), 1, None, H, None), INVALID, "bad raster size",
     True),
    ("check_accumulation_short_ld_fdr", "ofl_check_accumulation_u8",
     lambda b: acc(b, H, ld_fdr=C - 1, check=True), INVALID, "leading dimension", False),
    ("check_accumulation_device_short_ld_fac", "ofl_check_accumulation_u8",
     lambda b: acc(b, D, ld_fac=C - 1, check=True), INVALID, "leading dimension", False),
    ("check_accumulation_null_n_bad", "ofl_check_accumulation_u8",
     lambda b: acc(b, H, check=True, n_bad=ctypes.POINTER(ctypes.c_int64)()), INVALID, "null result pointer", False),
    ("strip_check_short_ld_fdr", "ofl_strip_check_accumulation_u8",
     lambda b: (b.dev((R + 2) * C), R, C, C - 1, b.dev(8 * R * C), C, None, None, i64(), None), INVALID,
     "leading dimension", False),
    ("flat_edges_null_edges", "ofl_flat_edges_f32",
     lambda b: (b.host(4 * R * C), b.host(R * C), R, C, None, i64(), i64(), H, None), INVALID, "null raster pointer",
     False),
    ("flat_edges_unknown_mem_kind", "ofl_flat_edges_f32",
     lambda b: (b.host(4 * R * C), b.host(R * C), R, C, b.host(R * C), i64(), i64(), 3, None), INVALID,
     "unknown mem_kind", False),
    ("resolve_flats_host_small_workspace", "ofl_resolve_flats_f32",
     lambda b: flats(b, H, work=True), WORKSPACE, "workspace too small", False),
    ("resolve_flats_host_null_mask", "ofl_resolve_flats_f32",
     lambda b: flats(b, H, flat_mask=True), INVALID, "null raster pointer", False),
    ("resolve_flats_over_2_32_cells", "ofl_resolve_flats_f32",
     lambda b: (b.host(4), b.host(1), BIG, BIG // 2, b.host(4), b.host(4), i64(5), None, 0, H, None), INVALID,
     "at most 2^32 cells", True),
    ("fix_flats_device_null_mask", "ofl_fix_flats_f32",
     lambda b: flats(b, D, flat_mask=True), INVALID, "null raster pointer", False),
    ("masked_dirs_null_labels", "ofl_d8_masked_flow_dirs_i32",
     lambda b: (b.host(4 * R * C), None, b.host(R * C), R, C, H, None), INVALID, "null raster pointer", False),
    ("flat_gradient_too_many_seeds", "ofl_flat_gradient_i32",
     lambda b: (b.host(4 * R * C), b.host(R * C), R, C, b.host(4 * (R * C + 1)), R * C + 1, 0, b.host(4 * R * C),
                None, 0, None, 0, H, None), INVALID, "count out of range", False),
    ("flat_gradient_null_seeds", "ofl_flat_gradient_i32",
     lambda b: (b.host(4 * R * C), b.host(R * C), R, C, None, 3, 0, b.host(4 * R * C), None, 0, None, 0, H, None),
     INVALID, "null raster pointer", False),
    ("pits_host_small_workspace", "ofl_breach_single_cell_pits_f32",
     lambda b: (b.host(4 * R * C), R, C, C, -9999.0, b.host(R * C), i64(3), b.dev(16), 16, H, None), WORKSPACE,
     "workspace too small", False),
    ("pits_short_ld", "ofl_breach_single_cell_pits_f32",
     lambda b: (b.host(4 * R * C), R, C, C - 1, -9999.0, b.host(R * C), i64(3), None, 0, H, None), INVALID,
     "leading dimension", False),
    ("pits_over_2_32_cells", "ofl_breach_single_cell_pits_f32",
     lambda b: (b.host(4), BIG, BIG // 2, BIG // 2, -9999.0, b.host(1), i64(3), None, 0, H, None), INVALID,
     "at most 2^32 cells", True),
    ("strip_local_negative_cols", "ofl_strip_accum_local",
     lambda b: strip_local(b, cols=-1, ld=1), INVALID, "bad raster size", False),
    ("strip_local_small_workspace", "ofl_strip_accum_local",
     lambda b: strip_local(b, work=16), WORKSPACE, "workspace too small", False),
    ("strip_local_one_row", "ofl_strip_accum_local",
     lambda b: strip_local(b, rows=1), INVALID, "at least 2 rows", False),
    ("strip_local_rows_not_tile_multiple", "ofl_strip_accum_local",
     lambda b: strip_local(b, rows=R + 3, has_below=1), INVALID, "multiple of", False),
    ("strip_boundary_no_strips", "ofl_strip_boundary_solve",
     lambda b: (b.dev(1 << 16), 0, C, b.dev(1 << 16), b.dev(1 << 16), 1 << 16, None), INVALID,
     "bad boundary graph size", False),
    ("strip_boundary_small_workspace", "ofl_strip_boundary_solve",
     lambda b: (b.dev(1 << 16), 2, C, b.dev(1 << 16), b.dev(16), 16, None), WORKSPACE, "workspace too small", False),
    ("strip_final_null_j", "ofl_strip_accum_final",
     lambda b: (b.dev((R + 2) * C), R, C, C, 0, 0, None, b.dev(1 << 20), 1 << 20, b.dev(8 * R * C), C, None), INVALID,
     "null raster pointer", False),
    ("strip_collect_null_flags", "ofl_strip_collect_flags",
     lambda b: (b.dev(1 << 20), R, C, None, 0, None, None), INVALID, "null pointer", False),
    ("basins_host_small_workspace", "ofl_label_basins_u8",
     lambda b: (b.host(R * C), R, C, C, None, 0, b.host(8 * R * C), C, b.dev(16), 16, H, None), WORKSPACE,
     "workspace too small", False),
    ("basins_negative_pour_count", "ofl_label_basins_u8",
     lambda b: (b.host(R * C), R, C, C, None, -1, b.host(8 * R * C), C, None, 0, H, None), INVALID,
     "pour-point count", False),
    ("basins_null_pour_points", "ofl_label_basins_u8",
     lambda b: (b.host(R * C), R, C, C, None, 2, b.host(8 * R * C), C, None, 0, H, None), INVALID,
     "null raster pointer", False),
    ("basins_device_short_ld_labels", "ofl_label_basins_u8",
     lambda b: (b.dev(R * C), R, C, C, None, 0, b.dev(8 * R * C), C - 1, None, 0, D, None), INVALID,
     "leading dimension", False),
    ("basins_too_large", "ofl_label_basins_u8",
     lambda b: (b.host(1), 1 << 30, 1, 1, None, 0, b.host(8), 1, None, 0, H, None), INVALID, "bad raster size", True),
    ("check_basins_null_n_bad", "ofl_check_basins_u8",
     lambda b: (b.host(R * C), R, C, C, None, 0, b.host(8 * R * C), C, None, H, None), INVALID, "null result pointer",
     False),
    ("synth_unknown_kind", "ofl_synth_dem_f32",
     lambda b: (b.dev(4 * R * C), R, C, C, 0, R, 1, 9, 1.0, 0, -9999.0, None), INVALID, "unknown synthetic DEM kind",
     False),
    ("synth_empty_short_ld", "ofl_synth_dem_f32",
     lambda b: (b.dev(1), 0, C, C - 1, 0, 0, 1, 0, 1.0, 0, -9999.0, None), INVALID, "leading dimension", False),
    ("synth_null_dem", "ofl_synth_dem_f32",
     lambda b: (None, R, C, C, 0, R, 1, 0, 1.0, 0, -9999.0, None), INVALID, "null raster pointer", False),
]


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _native.lib()


@pytest.fixture(scope="module")
def devices(lib):
    """(the library has a device, torch has one).  The library asks the CUDA runtime itself, so the two can differ."""
    import torch

    return lib.ofl_init(0) == 0, torch.cuda.is_available()


def test_every_compute_entry_point_has_a_case():
    compute = {n for n, (res, _) in _native.SIGNATURES.items() if res is ctypes.c_int} - {
        "ofl_abi_version", "ofl_init", "ofl_shutdown", "ofl_phase_timing_read"}
    assert compute == {c[1] for c in CASES}


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_bad_argument_is_refused_before_the_device(lib, devices, case):
    _, name, args, status, message, claims_more = case
    lib_device, torch_device = devices
    if claims_more and (lib_device or torch_device):
        pytest.skip("claims more memory than it passes: run only without a device")
    if lib_device and not torch_device:
        pytest.skip("the library has a device but torch cannot allocate on it")
    b = Buffers(torch_device)
    call_args = args(b)
    before = lib.ofl_launch_count()
    rc = getattr(lib, name)(*call_args)
    msg = lib.ofl_last_error().decode()
    assert (rc, message in msg) == (status, True), msg
    assert lib.ofl_launch_count() == before


def test_refused_call_zeroes_its_results(lib):
    n_low, n_high, n_bad = i64(), i64(), i64()
    n_low[0] = n_high[0] = n_bad[0] = 7
    assert lib.ofl_flat_edges_f32(None, None, R, C, None, n_low, n_high, H, None) == INVALID
    assert lib.ofl_check_basins_u8(None, R, C, C, None, 0, None, C, n_bad, 9, None) == INVALID
    assert (n_low[0], n_high[0], n_bad[0]) == (0, 0, 0)
