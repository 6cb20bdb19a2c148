"""ctypes binding of include/daisyworld_b200.h.  No fallback: if the CUDA library is missing or no
CUDA device is usable, importing works but creating an environment raises."""
import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DW_LIB", os.path.join(PKG, "libdaisyworld_b200.so"))   # DW_LIB: another build, e.g. to compare two

DW_POLICY = {"none": 0, "greedy": 1, "antigreedy": 2, "replay": 3, "random": 4, "eps_greedy": 5, "mlp": 6}
DW_E_UNSUPPORTED = -3       # include/daisyworld_b200.h: configuration outside what the kernels implement
DW_DIAG = {"temp": 0, "temp_light": 1, "temp_dark": 2, "temp_effective": 3, "beta": 4, "beta_l": 5, "beta_d": 6,
           "growth": 7}
# dwt_pool field selectors (include/daisyworld_b200_tiled.h): the diagnostics, the growth planes and grid channels 0-3, 5
DWT_FIELD = {"temp": 0, "temp_light": 1, "temp_dark": 2, "temp_effective": 3, "beta": 4, "beta_l": 5, "beta_d": 6,
             "growth_l": 7, "growth_d": 8, "grid_bare": 9, "grid_light": 10, "grid_dark": 11, "grid_temp": 12,
             "grid_temp_dark": 13}


class DwConfig(C.Structure):
    _fields_ = [("batch", C.c_int32), ("dim", C.c_int32), ("n_agents", C.c_int32), ("device", C.c_int32)] + \
               [(k, C.c_double) for k in ("p", "g", "S", "sigma", "gamma", "q", "q2", "temp_optimal", "dt", "agent_gamma",
                                          "albedo_bare", "albedo_light", "albedo_dark")] + \
               [("daisy_kernel", C.c_double * 9), ("adjacent_kernel", C.c_double * 9), ("obs_mask", C.c_double * 9)]


class DwClock(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("L", "dL", "min_L", "max_L", "ddL")] + \
               [("step_count", C.c_int64), ("ramp_period", C.c_int64), ("ramp_up_down", C.c_int32), ("_pad", C.c_int32)]


class DwProfile(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("fused_launches", C.c_uint64), ("fused_cell_updates", C.c_uint64),
                ("fused_ms", C.c_double)]


class DwRunResult(C.Structure):
    _fields_ = [("steps_run", C.c_int64), ("worlds_alive", C.c_int64), ("all_done_hit", C.c_int32), ("_pad", C.c_int32)]


# every symbol include/daisyworld_b200.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = [
    "dw_abi_version", "dw_last_error", "dw_create", "dw_destroy", "dw_set_config", "dw_set_clock", "dw_get_clock", "dw_get_last_L",
    "dw_set_stream", "dw_set_epsilon", "dw_set_mlp", "dw_set_mlp_population", "dw_run_population", "dw_get_population_results",
    "dw_upload_state", "dw_upload_covers", "dw_init_random", "dw_init_temperatures", "dw_set_profiling", "dw_get_profile", "dw_step_out_layout", "dw_step_packed", "dw_host_alloc", "dw_host_free", "dw_update_agents",
    "dw_agents_begin", "dw_agents_collide", "dw_step_tail_packed", "dw_step_tail_counted",
    "dw_forward", "dw_get_obs_at", "dw_get_grid", "dw_trim_supported", "dw_run_chunk_masked", "dw_trim_lifespans", "dw_get_grid_f32", "dw_get_obs_f32", "dw_f32_stats", "dw_debug_time_materialise", "dw_get_agents", "dw_get_obs", "dw_get_diag", "dw_get_diag_stats", "dw_get_cover_stats",
    "dw_run", "dw_run_chunk", "dw_run_series", "dw_reset_lifespans", "dw_get_lifespans", "dw_lifespan_stats_device",
    "dw_checkpoint_save", "dw_checkpoint_restore", "dw_synchronize", "dw_set_world_offset", "dw_debug_slow_count", "dw_debug_state",
    "dw_debug_root4", "dw_debug_markstein", "dw_debug_markstein_f32", "dw_debug_fp64_peak", "dw_debug_screen_error",
]

# every symbol include/daisyworld_b200_tiled.h declares (single giant grid, row bands)
TILED_SYMBOLS = [
    "dwt_last_error", "dwt_create", "dwt_destroy", "dwt_set_config", "dwt_set_clock", "dwt_get_clock", "dwt_set_stream", "dwt_set_epsilon",
    "dwt_synchronize", "dwt_upload_covers", "dwt_upload_agents", "dwt_init_random", "dwt_decide", "dwt_move_graze",
    "dwt_finish_agents", "dwt_stencil", "dwt_halo_wrap", "dwt_get_ptrs", "dwt_run", "dwt_end_chunk",
    "dwt_reset_lifespans", "dwt_get_lifespans", "dwt_get_agents", "dwt_get_covers", "dwt_get_grid",
    "dwt_debug_slow_count", "dwt_debug_time_stencil", "dwt_cover_checksum", "dwt_ipc_export", "dwt_ipc_attach", "dwt_get_peer_buffers", "dwt_attach_peers", "dwt_step_p2p",
    "dwt_flush_p2p", "dwt_peer_status", "dwt_set_series", "dwt_get_series_ptr", "dwt_get_series", "dwt_get_pitch", "dwt_set_peer_rows",
    "dwt_observe", "dwt_get_obs_ptr", "dwt_get_obs", "dwt_set_mlp",
    "dwt_get_diag", "dwt_get_diag_stats", "dwt_get_cover_stats", "dwt_pool", "dwt_get_pool_ptr", "dwt_get_pool", "dwt_get_last_L",
    "dwt_save_state", "dwt_restore_state", "dwt_pre_checksum",
    "dwt_grid_f32", "dwt_get_grid_f32_ptr", "dwt_get_grid_f32", "dwt_f32_stats", "dwt_debug_time_materialise",
]


# representations of a band's state in a snapshot (dwt_band_state)
DWT_REP = {"none": 0, "planes": 1, "lattice": 2}


class DwtBandState(C.Structure):
    _fields_ = [("cur_rep", C.c_int32), ("pre_rep", C.c_int32), ("L_last", C.c_double), ("done_at", C.c_int64),
                ("cur_bytes", C.c_uint64), ("pre_bytes", C.c_uint64)]


class DwtPtrs(C.Structure):
    _fields_ = [("act", C.c_void_p), ("gain", C.c_void_p), ("stepmax", C.c_void_p), ("send_top", C.c_void_p),
                ("send_bottom", C.c_void_p), ("recv_top", C.c_void_p), ("recv_bottom", C.c_void_p)]


_lib = None


class DaisyWorldError(RuntimeError):
    pass


def load():
    """Load the C-ABI library; raises if it has not been built (python -m therldaisyworld_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DaisyWorldError(f"{LIB_PATH} not found: build it with `python -m therldaisyworld_b200.build` "
                              "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    pd, pi64, pu8, pi8 = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_uint8), C.POINTER(C.c_int8)
    sig = {
        "dw_abi_version": (C.c_int, []),
        "dw_last_error": (C.c_char_p, [vp]),
        "dw_create": (C.c_int, [C.POINTER(DwConfig), C.POINTER(vp)]),
        "dw_destroy": (C.c_int, [vp]),
        "dw_set_config": (C.c_int, [vp, C.POINTER(DwConfig)]),
        "dw_set_clock": (C.c_int, [vp, C.POINTER(DwClock)]),
        "dw_get_clock": (C.c_int, [vp, C.POINTER(DwClock)]),
        "dw_get_last_L": (C.c_int, [vp, pd]),
        "dw_set_stream": (C.c_int, [vp, vp]),
        "dw_set_epsilon": (C.c_int, [vp, C.c_double]),
        "dw_set_mlp": (C.c_int, [vp, pd, i32]),
        "dw_set_mlp_population": (C.c_int, [vp, pd, i32, i32]),
        "dw_run_population": (C.c_int, [vp, i64, pi64]),
        "dw_get_population_results": (C.c_int, [vp, pd, pi64, pi64]),
        "dw_upload_state": (C.c_int, [vp, pd, pi64, pd]),
        "dw_upload_covers": (C.c_int, [vp, pd, pd]),
        "dw_init_random": (C.c_int, [vp, u64, C.c_double, C.c_double, C.c_double, C.c_double]),
        "dw_init_temperatures": (C.c_int, [vp]),
        "dw_set_profiling": (C.c_int, [vp, i32]),
        "dw_get_profile": (C.c_int, [vp, C.POINTER(DwProfile)]),
        "dw_step_out_layout": (C.c_int, [vp, pi64]),
        "dw_step_packed": (C.c_int, [vp, pi64, i32, i32, i32, u64, i32, vp, C.POINTER(DwClock)]),
        "dw_host_alloc": (C.c_int, [u64, C.POINTER(vp)]),
        "dw_host_free": (C.c_int, [vp]),
        "dw_update_agents": (C.c_int, [vp, pi64, i32, i32]),
        "dw_agents_begin": (C.c_int, [vp, pi64, i32, i32, i32, u64, pi64]),
        "dw_agents_collide": (C.c_int, [vp, pd, C.POINTER(C.c_int32), C.c_double]),
        "dw_step_tail_packed": (C.c_int, [vp, i32, vp, C.POINTER(DwClock)]),
        "dw_step_tail_counted": (C.c_int, [vp, C.POINTER(C.c_int64)]),
        "dw_forward": (C.c_int, [vp, pd, pd]),
        "dw_get_obs_at": (C.c_int, [vp, pi64, i32, i32, pd]),
        "dw_get_grid": (C.c_int, [vp, pd]),
        "dw_get_grid_f32": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "dw_get_obs_f32": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "dw_f32_stats": (C.c_int, [vp, C.POINTER(C.c_uint64)]),
        "dw_trim_supported": (C.c_int, [vp, C.c_int32, C.POINTER(C.c_int32)]),
        "dw_run_chunk_masked": (C.c_int, [vp, C.c_int32, C.c_int32, C.POINTER(C.c_int8), C.c_uint64, C.POINTER(C.c_uint64)]),
        "dw_trim_lifespans": (C.c_int, [vp, C.c_int32]),
        "dw_debug_time_materialise": (C.c_int, [vp, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
        "dw_get_agents": (C.c_int, [vp, pi64, pd]),
        "dw_get_obs": (C.c_int, [vp, pd]),
        "dw_get_diag": (C.c_int, [vp, i32, pd]),
        "dw_get_diag_stats": (C.c_int, [vp, i32, pd]),
        "dw_get_cover_stats": (C.c_int, [vp, pd]),
        "dw_run": (C.c_int, [vp, i64, i32, pi8, u64, i32, C.POINTER(DwRunResult)]),
        "dw_run_chunk": (C.c_int, [vp, i32, i32, pi8, u64, C.POINTER(u64)]),
        "dw_run_series": (C.c_int, [vp, i64, i32, pi8, u64, pd]),
        "dw_reset_lifespans": (C.c_int, [vp]),
        "dw_get_lifespans": (C.c_int, [vp, pi64, pi64]),
        "dw_lifespan_stats_device": (C.c_int, [vp, vp]),
        "dw_checkpoint_save": (C.c_int, [vp]),
        "dw_checkpoint_restore": (C.c_int, [vp]),
        "dw_synchronize": (C.c_int, [vp]),
        "dw_set_world_offset": (C.c_int, [vp, C.c_uint32]),
        "dw_debug_slow_count": (C.c_int, [vp, C.POINTER(u64), i32]),
        "dw_debug_state": (C.c_int, [vp, C.POINTER(C.c_int32)]),
        "dw_debug_root4": (C.c_int, [vp, pd, pd, i32]),
        "dw_debug_screen_error": (C.c_int, [vp, pd, pd]),
        "dw_debug_markstein": (C.c_int, [vp, C.c_uint32, C.POINTER(C.c_uint32)]),
        "dw_debug_markstein_f32": (C.c_int, [vp, C.c_uint32, C.POINTER(C.c_uint32)]),
        "dw_debug_fp64_peak": (C.c_int, [vp, i32, i32, pd, pd]),
    }
    assert set(sig) == set(SYMBOLS)
    pi32 = C.POINTER(C.c_int32)
    tsig = {
        "dwt_last_error": (C.c_char_p, [vp]),
        "dwt_create": (C.c_int, [C.POINTER(DwConfig), i32, i32, i32, C.POINTER(vp)]),
        "dwt_destroy": (C.c_int, [vp]),
        "dwt_set_config": (C.c_int, [vp, C.POINTER(DwConfig)]),
        "dwt_set_clock": (C.c_int, [vp, C.POINTER(DwClock)]),
        "dwt_get_clock": (C.c_int, [vp, C.POINTER(DwClock)]),
        "dwt_set_stream": (C.c_int, [vp, vp]),
        "dwt_set_epsilon": (C.c_int, [vp, C.c_double]),
        "dwt_synchronize": (C.c_int, [vp]),
        "dwt_upload_covers": (C.c_int, [vp, pd, pd]),
        "dwt_upload_agents": (C.c_int, [vp, pi64, pd]),
        "dwt_init_random": (C.c_int, [vp, u64, C.c_double, C.c_double, C.c_double, C.c_double]),
        "dwt_decide": (C.c_int, [vp, i32, pi8, u64]),
        "dwt_move_graze": (C.c_int, [vp]),
        "dwt_finish_agents": (C.c_int, [vp]),
        "dwt_stencil": (C.c_int, [vp, i32]),
        "dwt_halo_wrap": (C.c_int, [vp]),
        "dwt_get_ptrs": (C.c_int, [vp, C.POINTER(DwtPtrs)]),
        "dwt_run": (C.c_int, [vp, i64, i32, pi8, u64]),
        "dwt_end_chunk": (C.c_int, [vp, i32, pi32]),
        "dwt_reset_lifespans": (C.c_int, [vp]),
        "dwt_get_lifespans": (C.c_int, [vp, pi64, pi64]),
        "dwt_get_agents": (C.c_int, [vp, pi64, pd]),
        "dwt_get_covers": (C.c_int, [vp, pd, pd]),
        "dwt_get_grid": (C.c_int, [vp, pd]),
        "dwt_debug_slow_count": (C.c_int, [vp, C.POINTER(u64)]),
        "dwt_cover_checksum": (C.c_int, [vp, C.POINTER(u64)]),
        "dwt_debug_time_stencil": (C.c_int, [vp, i32, pd]),
        "dwt_ipc_export": (C.c_int, [vp, vp]),
        "dwt_ipc_attach": (C.c_int, [vp, i32, i32, vp]),
        "dwt_get_peer_buffers": (C.c_int, [vp, C.POINTER(vp)]),
        "dwt_attach_peers": (C.c_int, [vp, i32, i32, C.POINTER(vp)]),
        "dwt_step_p2p": (C.c_int, [vp, i32, pi8, u64]),
        "dwt_flush_p2p": (C.c_int, [vp]),
        "dwt_peer_status": (C.c_int, [vp, pi32]),
        "dwt_set_series": (C.c_int, [vp, i32]),
        "dwt_get_series_ptr": (C.c_int, [vp, C.POINTER(vp)]),
        "dwt_get_series": (C.c_int, [vp, i32, pd]),
        "dwt_get_pitch": (C.c_int, [vp, pi32]),
        "dwt_set_peer_rows": (C.c_int, [vp, i32, pi32]),
        "dwt_observe": (C.c_int, [vp]),
        "dwt_get_obs_ptr": (C.c_int, [vp, C.POINTER(vp)]),
        "dwt_get_obs": (C.c_int, [vp, pd]),
        "dwt_set_mlp": (C.c_int, [vp, pd, i32]),
        "dwt_get_diag": (C.c_int, [vp, i32, pd]),
        "dwt_get_diag_stats": (C.c_int, [vp, i32, pd]),
        "dwt_get_cover_stats": (C.c_int, [vp, pd]),
        "dwt_pool": (C.c_int, [vp, i32, i32]),
        "dwt_get_pool_ptr": (C.c_int, [vp, C.POINTER(vp), pi32]),
        "dwt_get_pool": (C.c_int, [vp, pd]),
        "dwt_get_last_L": (C.c_int, [vp, pd]),
        "dwt_save_state": (C.c_int, [vp, C.POINTER(DwtBandState), vp, vp, pi64]),
        "dwt_restore_state": (C.c_int, [vp, C.POINTER(DwtBandState), vp, vp, pi64]),
        "dwt_pre_checksum": (C.c_int, [vp, C.POINTER(u64)]),
        "dwt_grid_f32": (C.c_int, [vp]),
        "dwt_get_grid_f32_ptr": (C.c_int, [vp, C.POINTER(vp)]),
        "dwt_get_grid_f32": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "dwt_f32_stats": (C.c_int, [vp, C.POINTER(u64)]),
        "dwt_debug_time_materialise": (C.c_int, [vp, i32, i32, pd]),
    }
    assert set(tsig) == set(TILED_SYMBOLS)
    sig.update(tsig)
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)      # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.dw_abi_version() != 3:
        raise DaisyWorldError("ABI version mismatch between _lib.py and libdaisyworld_b200.so")
    _lib = lib
    return lib


def check_tiled(lib, handle, rc, what):
    if rc != 0:
        msg = lib.dwt_last_error(handle)
        raise DaisyWorldError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def check(lib, handle, rc, what):
    if rc != 0:
        msg = lib.dw_last_error(handle)
        raise DaisyWorldError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
