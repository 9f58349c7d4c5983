"""ctypes binding of liboverflow_b200.so (include/overflow_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is usable,
every compute call raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liboverflow_b200.so")

OFL_MEM_HOST = 0
OFL_MEM_DEVICE = 1
OFL_DIR_MODE_TILE = 0
OFL_DIR_MODE_RASTER = 1
OFL_DIR_MODE_STRIP = 2

OFL_ELEM_F64 = 0
OFL_ELEM_I64 = 1
OFL_ELEM_U64 = 2

OFL_ERR_INVALID = -1
OFL_ERR_CYCLE = -5
OFL_ERR_WORKSPACE = -6


class OverflowB200Error(RuntimeError):
    """A liboverflow_b200 call failed (status code in .status)."""

    def __init__(self, status, message):
        super().__init__(f"liboverflow_b200 error {status}: {message}")
        self.status = status


_lib = None

# every symbol include/overflow_b200.h declares, with its ctypes signature
_i64, _f64, _vp, _int, _sz = ctypes.c_int64, ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
SIGNATURES = {
    "ofl_last_error": (ctypes.c_char_p, []),
    "ofl_abi_version": (_int, []),
    "ofl_init": (_int, [_int]),
    "ofl_shutdown": (_int, []),
    "ofl_launch_count": (_i64, []),
    "ofl_launch_count_reset": (None, []),
    "ofl_phase_timing_enable": (None, [_int]),
    "ofl_phase_timing_read": (_int, [ctypes.POINTER(_f64), ctypes.POINTER(_i64), _int, _int]),
    "ofl_flow_direction_f32": (_int, [_vp, _i64, _i64, _i64, _f64, _vp, _i64, _int, _int, _vp]),
    "ofl_flow_direction_x64": (_int, [_vp, _int, _i64, _i64, _i64, _f64, _vp, _i64, _int, _int, _vp]),
    "ofl_perimeter_count": (_i64, [_i64, _i64]),
    "ofl_accumulation_workspace_bytes": (_sz, [_i64, _i64]),
    "ofl_flow_accumulation_u8": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _sz, _int, _vp]),
    "ofl_flow_accumulation_seeded_u8": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _sz, _int, _vp]),
    "ofl_flow_routing_f32": (_int, [_vp, _i64, _i64, _i64, _f64, _vp, _i64, _vp, _i64, _vp, _int, _vp]),
    "ofl_check_accumulation_u8": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, ctypes.POINTER(_i64), _int, _vp]),
    "ofl_strip_check_accumulation_u8": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp, ctypes.POINTER(_i64), _vp]),
    "ofl_fill_border_u8": (_int, [_vp, _i64, _i64, _i64, _int, _vp]),
    "ofl_strip_workspace_bytes": (_sz, [_i64, _i64]),
    "ofl_strip_boundary_workspace_bytes": (_sz, [_int, _i64]),
    "ofl_strip_record_bytes": (_sz, [_i64]),
    "ofl_strip_accum_local": (_int, [_vp, _i64, _i64, _i64, _int, _int, _vp, _i64, _vp, _sz, _vp, _vp]),
    "ofl_strip_boundary_solve": (_int, [_vp, _int, _i64, _vp, _vp, _sz, _vp]),
    "ofl_strip_collect_flags": (_int, [_vp, _i64, _i64, _vp, _int, _vp, _vp]),
    "ofl_strip_accum_final": (_int, [_vp, _i64, _i64, _i64, _int, _int, _vp, _vp, _sz, _vp, _i64, _vp]),
    "ofl_flats_workspace_bytes": (_sz, [_i64, _i64]),
    "ofl_flat_edges_f32": (_int, [_vp, _vp, _i64, _i64, _vp, ctypes.POINTER(_i64), ctypes.POINTER(_i64), _int, _vp]),
    "ofl_resolve_flats_f32": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, ctypes.POINTER(_i64), _vp, _sz, _int, _vp]),
    "ofl_flat_gradient_i32": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _int, _vp, _vp, _i64, _vp, _sz, _int, _vp]),
    "ofl_d8_masked_flow_dirs_i32": (_int, [_vp, _vp, _vp, _i64, _i64, _int, _vp]),
    "ofl_fix_flats_f32": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, ctypes.POINTER(_i64), _vp, _sz, _int, _vp]),
    "ofl_pits_workspace_bytes": (_sz, [_i64, _i64]),
    "ofl_breach_single_cell_pits_f32": (_int, [_vp, _i64, _i64, _i64, _f64, _vp, ctypes.POINTER(_i64), _vp, _sz, _int, _vp]),
    "ofl_basins_workspace_bytes": (_sz, [_i64, _i64]),
    "ofl_label_basins_u8": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _vp, _sz, _int, _vp]),
    "ofl_check_basins_u8": (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, ctypes.POINTER(_i64), _int, _vp]),
    "ofl_synth_dem_f32": (_int, [_vp, _i64, _i64, _i64, _i64, _i64, ctypes.c_uint64, _int, ctypes.c_float, _int,
                                 ctypes.c_float, _vp]),
}


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OverflowB200Error(
            -100,
            f"{LIB_PATH} not found: build it with `python -m overflow_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback.",
        )
    handle = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def check(status):
    if status != 0:
        msg = lib().ofl_last_error()
        raise OverflowB200Error(status, msg.decode("utf-8", "replace") if msg else "unknown error")


_current_device = None


def init(device=0):
    """Select the CUDA device for subsequent calls (cheap when it is already selected)."""
    global _current_device
    device = int(device)
    if _current_device != device:
        check(lib().ofl_init(device))
        _current_device = device


def launch_count():
    return int(lib().ofl_launch_count())


def launch_count_reset():
    lib().ofl_launch_count_reset()


PHASES = ("direction", "acc_tile_a", "acc_solve", "acc_tile_b", "acc_links", "strip_edge", "flats_stencils", "flats_label", "flats_sweeps", "breach_pits",
          "basins_tile", "basins_solve", "basins_final")


def phase_timing_enable(on=True):
    lib().ofl_phase_timing_enable(1 if on else 0)


def phase_timing_read(reset=True):
    """{phase: (total_ms, launches)} measured with CUDA events on the launching stream."""
    n = len(PHASES)
    ms = (_f64 * n)()
    cnt = (_i64 * n)()
    lib().ofl_phase_timing_read(ms, cnt, n, 1 if reset else 0)
    return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(PHASES)}
